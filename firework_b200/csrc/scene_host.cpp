#include "scene_host.h"

#include <charconv>

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <functional>

#include "../../include/firework_b200.h"
#include "yaml_lite.h"

namespace fw {

using fwyaml::Node;

// ------------------------------------------------------------------------------------------------------
// YAML -> SceneDesc
// ------------------------------------------------------------------------------------------------------
namespace {

struct Loader {
    SceneDesc& sc;
    std::string err;
    explicit Loader(SceneDesc& s) : sc(s) {}

    bool fail(const Node* n, const std::string& msg) {
        if (err.empty()) err = (n ? "line " + std::to_string(n->line) + ": " : std::string()) + msg;
        return false;
    }
    const Node* req(const Node& m, const char* key) {
        const Node* n = m.get(key);
        if (!n) fail(&m, std::string("missing field `") + key + "`");
        return n;
    }
    bool as_f32(const Node* n, float& out) {
        if (!n) return false;
        if (n->kind != Node::SCALAR) return fail(n, "expected a number");
        const std::string_view v = n->scalar;
        // the common case — a plain decimal — through from_chars (no locale, no copy); everything it does not take
        // whole (".inf", "+1", hex, ...) through the YAML spellings and strtod as before.  Both round correctly.
        {
            double d;
            auto r = std::from_chars(v.data(), v.data() + v.size(), d);
            if (r.ec == std::errc() && r.ptr == v.data() + v.size()) { out = (float)d; return true; }
        }
        const std::string s(v);
        if (s == ".nan" || s == ".NaN") { out = NAN; return true; }
        if (s == ".inf" || s == "+.inf") { out = INFINITY; return true; }
        if (s == "-.inf") { out = -INFINITY; return true; }
        char* end = nullptr;
        double d = strtod(s.c_str(), &end);
        if (end == s.c_str() || *end) return fail(n, "invalid number `" + s + "`");
        out = (float)d;
        return true;
    }
    bool as_u64(const Node* n, uint64_t& out) {
        if (!n) return false;
        if (n->kind != Node::SCALAR) return fail(n, "expected an integer");
        const std::string_view sv = n->scalar;
        {
            unsigned long long v;
            auto r = std::from_chars(sv.data(), sv.data() + sv.size(), v, 10);
            if (r.ec == std::errc() && r.ptr == sv.data() + sv.size()) { out = v; return true; }
        }
        const std::string s(sv);
        char* end = nullptr;
        if (!s.empty() && s[0] == '-') return fail(n, "expected a non-negative integer, got `" + s + "`");
        unsigned long long v = strtoull(s.c_str(), &end, 10);
        if (end == s.c_str() || *end) return fail(n, "invalid integer `" + s + "`");
        out = v;
        return true;
    }
    bool as_int(const Node* n, int& out) {
        uint64_t v;
        if (!as_u64(n, v)) return false;
        if (v > 0x7fffffffu) return fail(n, "integer out of range");
        out = (int)v;
        return true;
    }
    bool as_bool(const Node* n, bool& out) {
        if (!n) return false;
        if (n->kind == Node::SCALAR && (n->scalar == "true" || n->scalar == "false")) {
            out = n->scalar == "true";
            return true;
        }
        return fail(n, "expected true/false");
    }
    bool as_str(const Node* n, std::string& out) {
        if (!n) return false;
        if (n->kind != Node::SCALAR) return fail(n, "expected a string");
        out = std::string(n->scalar);
        return true;
    }
    bool as_v3(const Node* n, float out[3]) {
        if (!n) return false;
        if (n->kind != Node::MAP) return fail(n, "expected {x, y, z}");
        return as_f32(req(*n, "x"), out[0]) && as_f32(req(*n, "y"), out[1]) && as_f32(req(*n, "z"), out[2]);
    }
    bool as_v2(const Node* n, float out[2]) {
        if (!n) return false;
        if (n->kind != Node::MAP) return fail(n, "expected {x, y}");
        return as_f32(req(*n, "x"), out[0]) && as_f32(req(*n, "y"), out[1]);
    }
    int add_asset(const std::string& path, int kind) {
        for (size_t i = 0; i < sc.assets.size(); ++i)
            if (sc.assets[i].path == path && sc.assets[i].kind == kind) return (int)i;
        AssetDesc a;
        a.path = path;
        a.kind = kind;
        sc.assets.push_back(std::move(a));
        return (int)sc.assets.size() - 1;
    }

    // texture.rs — returns texture index or -1.  `level` is the texture's place on its root-to-leaf path (the root is 1).
    int texture(const Node* n, int level = 1) {
        if (!n) return -1;
        if (n->kind != Node::MAP) { fail(n, "expected a texture mapping"); return -1; }
        if (level > FW_MAX_TEXTURE_DEPTH) {
            fail(n, "texture tree deeper than " + std::to_string(FW_MAX_TEXTURE_DEPTH) + " levels: the renderer follows at most " +
                        std::to_string(FW_MAX_TEXTURE_DEPTH - 1) + " nested CheckerTextures over a leaf texture");
            return -1;
        }
        std::string tag;
        if (!as_str(req(*n, "texture"), tag)) return -1;
        TexRec t;
        memset(&t, 0, sizeof(t));
        if (tag == "ConstantTexture") {
            t.kind = TEX_CONSTANT;
            if (!as_v3(req(*n, "color"), t.color)) return -1;
        } else if (tag == "CheckerTexture") {
            t.kind = TEX_CHECKER;
            t.a = texture(req(*n, "odd"), level + 1);
            t.b = texture(req(*n, "even"), level + 1);
            if (t.a < 0 || t.b < 0) return -1;
            if (!as_f32(req(*n, "scale"), t.scale)) return -1;
        } else if (tag == "PerlinNoiseTexture") {
            t.kind = TEX_PERLIN;
            if (!as_f32(req(*n, "scale"), t.scale)) return -1;
        } else if (tag == "TurbulenceTexture" || tag == "MarbleTexture") {
            t.kind = tag == "TurbulenceTexture" ? TEX_TURBULENCE : TEX_MARBLE;
            uint64_t d;
            if (!as_u64(req(*n, "depth"), d) || !as_f32(req(*n, "scale"), t.scale)) return -1;
            t.depth = (int)std::min<uint64_t>(d, 1u << 20);
        } else if (tag == "ImageTexture") {
            t.kind = TEX_IMAGE;
            std::string path;
            if (!as_str(req(*n, "value"), path)) return -1;
            t.a = add_asset(path, 0);
        } else {
            fail(n, "unknown texture tag `" + tag + "`");
            return -1;
        }
        sc.texs.push_back(t);
        return (int)sc.texs.size() - 1;
    }

    // material.rs
    bool material(const Node& n) {
        std::string tag;
        if (!as_str(req(n, "material"), tag)) return false;
        MatRec m;
        memset(&m, 0, sizeof(m));
        m.tex = -1;
        if (tag == "LambertianMat" || tag == "EmissiveMat") {
            m.kind = tag == "LambertianMat" ? MAT_LAMBERTIAN : MAT_EMISSIVE;
            m.tex = texture(req(n, "albedo"));
            if (m.tex < 0) return false;
        } else if (tag == "IsotropicMat") {
            m.kind = MAT_ISOTROPIC;
            m.tex = texture(req(n, "texture"));
            if (m.tex < 0) return false;
        } else if (tag == "MetalMat") {
            m.kind = MAT_METAL;
            if (!as_v3(req(n, "albedo"), m.albedo) || !as_f32(req(n, "roughness"), m.param)) return false;
        } else if (tag == "DielectricMat") {
            m.kind = MAT_DIELECTRIC;
            if (!as_f32(req(n, "ref_idx"), m.param)) return false;
        } else {
            return fail(&n, "unknown material tag `" + tag + "`");
        }
        sc.mats.push_back(m);
        return true;
    }

    bool rect_fields(const Node& n, int plane, ShapeRec& s) {
        memset(&s, 0, sizeof(s));
        s.kind = SH_RECT;
        float mn[2], mx[2];
        bool flip;
        if (!as_v2(req(n, "min"), mn) || !as_v2(req(n, "max"), mx) || !as_f32(req(n, "k"), s.f[4]) ||
            !as_bool(req(n, "flip_normal"), flip) || !as_int(req(n, "material"), s.material))
            return false;
        s.f[0] = mn[0]; s.f[1] = mn[1]; s.f[2] = mx[0]; s.f[3] = mx[1];
        s.i0 = plane | (flip ? 4 : 0);
        return true;
    }
    static int plane_of(const std::string& tag) {
        if (tag == "XY" || tag == "XYRect") return 0;
        if (tag == "XZ" || tag == "XZRect") return 1;
        if (tag == "YZ" || tag == "YZRect") return 2;
        return -1;
    }

    // objects/*.rs — returns shape index or -1
    int shape(const Node* np) {
        if (!np) return -1;
        const Node& n = *np;
        if (n.kind != Node::MAP) { fail(np, "expected a shape mapping"); return -1; }
        std::string tag;
        if (!as_str(req(n, "object_type"), tag)) return -1;
        ShapeRec s;
        memset(&s, 0, sizeof(s));
        if (tag == "Sphere") {
            s.kind = SH_SPHERE;
            if (!as_f32(req(n, "radius"), s.f[0]) || !as_int(req(n, "material"), s.material)) return -1;
        } else if (plane_of(tag) >= 0) {
            if (!rect_fields(n, plane_of(tag), s)) return -1;
        } else if (tag == "Rect3d") {
            s.kind = SH_RECT3D;
            float pos[3], size[3];
            if (!as_v3(req(n, "pos"), pos) || !as_v3(req(n, "size"), size)) return -1;
            memcpy(&s.f[0], pos, 12);
            memcpy(&s.f[3], size, 12);
            const Node* faces = req(n, "faces");
            if (!faces) return -1;
            if (faces->kind != Node::SEQ && !faces->is_null()) { fail(faces, "expected a list of faces"); return -1; }
            std::vector<ShapeRec> fr;
            for (const Node& f : faces->children) {
                // enum Rect { XY(..), XZ(..), YZ(..) } — externally tagged: {XY: {...}}
                if (f.kind != Node::MAP || f.children.size() != 1) { fail(&f, "expected {XY|XZ|YZ: rect}"); return -1; }
                int plane = plane_of(std::string(f.children[0].key));
                if (plane < 0) { fail(&f, "unknown Rect variant `" + std::string(f.children[0].key) + "`"); return -1; }
                ShapeRec r;
                if (f.children[0].kind != Node::MAP) { fail(&f, "expected rect fields"); return -1; }
                if (!rect_fields(f.children[0], plane, r)) return -1;
                fr.push_back(r);
            }
            s.i0 = (int)sc.shapes.size();
            s.i1 = (int)fr.size();
            s.material = fr.empty() ? 0 : fr[0].material;
            for (auto& r : fr) sc.shapes.push_back(r);
        } else if (tag == "TriangleMesh") {
            s.kind = SH_MESH;
            MeshDesc m;
            const Node* idx = req(n, "indicies");
            const Node* verts = req(n, "verts");
            if (!idx || !verts) return -1;
            if (idx->kind != Node::SEQ || verts->kind != Node::SEQ) { fail(&n, "mesh needs indicies and verts lists"); return -1; }
            m.indicies.reserve(idx->children.size());
            for (const Node& i : idx->children) {
                uint64_t v;
                if (!as_u64(&i, v)) return -1;
                m.indicies.push_back((uint32_t)v);
            }
            m.verts.reserve(verts->children.size());
            for (const Node& v : verts->children) {
                float p[3];
                if (!as_v3(&v, p)) return -1;
                m.verts.push_back(V3{p[0], p[1], p[2]});
            }
            const Node* nn = n.get("normals");
            if (nn && nn->kind == Node::SEQ) {
                m.has_normals = true;
                for (const Node& v : nn->children) {
                    float p[3];
                    if (!as_v3(&v, p)) return -1;
                    m.normals.push_back(V3{p[0], p[1], p[2]});
                }
                if (m.normals.size() != m.verts.size()) { fail(nn, "TriangleMesh: normals.len() must equal verts.len()"); return -1; }
            }
            const Node* un = n.get("uvs");
            if (un && un->kind == Node::SEQ) {
                m.has_uvs = true;
                for (const Node& v : un->children) {
                    float p[2];
                    if (!as_v2(&v, p)) return -1;
                    m.uvs.push_back(p[0]);
                    m.uvs.push_back(p[1]);
                }
                if (m.uvs.size() != 2 * m.verts.size()) { fail(un, "TriangleMesh: uvs.len() must equal verts.len()"); return -1; }
            }
            if (!as_int(req(n, "material"), m.material)) return -1;
            if (m.indicies.size() < 3) { fail(&n, "TriangleMesh with no triangles"); return -1; }
            for (uint32_t i : m.indicies)
                if (i >= m.verts.size()) { fail(idx, "TriangleMesh index out of range"); return -1; }
            s.material = m.material;
            s.i0 = (int)sc.meshes.size();
            sc.meshes.push_back(std::move(m));
        } else if (tag == "Disk") {
            s.kind = SH_DISK;
            if (!as_f32(req(n, "radius"), s.f[0]) || !as_f32(req(n, "phi_max"), s.f[1]) ||
                !as_f32(req(n, "inner_radius"), s.f[2]) || !as_int(req(n, "material"), s.material))
                return -1;
        } else if (tag == "Cylinder") {
            s.kind = SH_CYLINDER;
            if (!as_f32(req(n, "radius"), s.f[0]) || !as_f32(req(n, "height"), s.f[1]) ||
                !as_f32(req(n, "max_phi"), s.f[2]) || !as_int(req(n, "material"), s.material))
                return -1;
        } else if (tag == "Cone") {
            s.kind = SH_CONE;
            if (!as_f32(req(n, "radius"), s.f[0]) || !as_f32(req(n, "height"), s.f[1]) ||
                !as_int(req(n, "material"), s.material))
                return -1;
        } else if (tag == "ConstantMedium") {
            s.kind = SH_MEDIUM;
            int inner = shape(req(n, "obj"));
            if (inner < 0) return -1;
            if (sc.shapes[inner].kind == SH_MEDIUM) { fail(&n, "nested ConstantMedium is not supported"); return -1; }
            s.i0 = inner;
            if (!as_f32(req(n, "density"), s.f[0]) || !as_int(req(n, "material"), s.material)) return -1;
        } else {
            fail(&n, "unknown object_type `" + tag + "`");
            return -1;
        }
        sc.shapes.push_back(s);
        return (int)sc.shapes.size() - 1;
    }

    bool object(const Node& n) {
        if (n.kind != Node::MAP) return fail(&n, "expected a render object mapping");
        ObjectDesc o;
        o.shape = shape(req(n, "obj"));
        if (o.shape < 0) return false;
        float p[3];
        if (!as_v3(req(n, "position"), p)) return false;
        o.position = V3{p[0], p[1], p[2]};
        const Node* rot = req(n, "rotation");
        if (!rot) return false;
        const Node* bv = req(*rot, "bv");
        if (!bv) return false;
        if (!as_f32(req(*rot, "s"), o.rotor[0]) || !as_f32(req(*bv, "xy"), o.rotor[1]) ||
            !as_f32(req(*bv, "xz"), o.rotor[2]) || !as_f32(req(*bv, "yz"), o.rotor[3]))
            return false;
        if (!as_bool(req(n, "flip_normals"), o.flip_normals)) return false;
        sc.objects.push_back(o);
        return true;
    }

    bool run(const Node& root) {
        if (root.kind != Node::MAP) return fail(&root, "scene document must be a mapping");
        const Node* mats = req(root, "materials");
        const Node* objs = req(root, "render_objects");
        const Node* env = req(root, "environment");
        if (!mats || !objs || !env) return false;
        if (mats->kind == Node::SEQ)
            for (const Node& m : mats->children)
                if (!material(m)) return false;
        if (objs->kind == Node::SEQ)
            for (const Node& o : objs->children)
                if (!object(o)) return false;
        // validate material indices (the reference would panic on use: scene.rs:86)
        for (const ShapeRec& s : sc.shapes)
            if (s.kind != SH_RECT3D && (s.material < 0 || s.material >= (int)sc.mats.size()))
                return fail(objs, "shape refers to material " + std::to_string(s.material) + " but the scene has " +
                                      std::to_string(sc.mats.size()));
        std::string tag;
        if (env->kind != Node::MAP || !as_str(req(*env, "environment"), tag)) return fail(env, "bad environment");
        if (tag == "ColorEnv") {
            sc.env_kind = ENV_COLOR;
            if (!as_v3(req(*env, "color"), sc.env_a)) return false;
        } else if (tag == "SkyEnv") {
            sc.env_kind = ENV_SKY;
            if (!as_v3(req(*env, "zenith_color"), sc.env_a) || !as_v3(req(*env, "horizon_color"), sc.env_b)) return false;
        } else if (tag == "HdrEnvironment") {
            sc.env_kind = ENV_HDR;
            std::string path;
            if (!as_str(req(*env, "value"), path)) return false;
            sc.env_asset = add_asset(path, 1);
        } else {
            return fail(env, "unknown environment tag `" + tag + "`");
        }
        return true;
    }
};

}  // namespace

bool load_scene_yaml(const char* text, size_t len, SceneDesc& out, std::string& err) {
    Node root;
    if (!fwyaml::parse(text, len, root, err)) return false;
    out = SceneDesc();
    Loader ld(out);
    if (!ld.run(root)) {
        err = ld.err.empty() ? "invalid scene document" : ld.err;
        return false;
    }
    return true;
}

// ------------------------------------------------------------------------------------------------------
// f32 helpers with the reference's operation order (ultraviolet Vec3 / Mat3, aabb.rs)
// ------------------------------------------------------------------------------------------------------
static inline V3 vmin(V3 a, V3 b) { return V3{fminf(a.x, b.x), fminf(a.y, b.y), fminf(a.z, b.z)}; }
static inline V3 vmax(V3 a, V3 b) { return V3{fmaxf(a.x, b.x), fmaxf(a.y, b.y), fmaxf(a.z, b.z)}; }
static inline Box box_expand(const Box& a, const Box& b) { return Box{vmin(a.mn, b.mn), vmax(a.mx, b.mx)}; }  // aabb.rs:52
static inline float comp(const V3& v, int i) { return i == 0 ? v.x : (i == 1 ? v.y : v.z); }
static inline V3 box_center(const Box& b) {  // aabb.rs:59-61
    return V3{0.5f * b.mn.x + 0.5f * b.mx.x, 0.5f * b.mn.y + 0.5f * b.mx.y, 0.5f * b.mn.z + 0.5f * b.mx.z};
}

// ------------------------------------------------------------------------------------------------------
// BVH build: bvh.rs:21-71, in three stages: (a) the reference's median-split tree, which fixes the leaves;
// (b) an SAH interior over those leaves; (c) the collapse into 4-wide nodes.  (a) and (b) run on the host or,
// for large trees, on a CUDA device (kernels_build.cu); (c) is shared.
// ------------------------------------------------------------------------------------------------------
namespace {
struct BuildNode {
    Box box;
    int left = -1, right = -1;  // interior
    int first = -1, count = 0;  // leaf: range in the ordered item list
    int depth = 0;
    bool unbounded = false;     // some item below has a box that does not bound its geometry
};
// fminf / fmaxf as glibc computes them on x86-64 (minss / maxss plus its NaN path): a quiet NaN operand loses, two quiet
// NaNs give the first, a signaling NaN gives a + b, and a tie (-0.0 against +0.0) gives the SECOND operand.  Spelled out
// for the node boxes because a compiler may swap the operands of a call it knows to be commutative, and the signs of zero
// in those boxes are part of the flattened tree.
static inline bool is_snan(float x) {
    uint32_t u;
    memcpy(&u, &x, 4);
    return (u & 0x7fc00000u) == 0x7f800000u && (u & 0x003fffffu) != 0;
}
static inline float lib_min(float a, float b) {
    return a < b ? a : b < a ? b : (is_snan(a) || is_snan(b)) ? a + b : a != a ? (b != b ? a : b) : b != b ? a : b;
}
static inline float lib_max(float a, float b) {
    return a > b ? a : b > a ? b : (is_snan(a) || is_snan(b)) ? a + b : a != a ? (b != b ? a : b) : b != b ? a : b;
}
// The median-split tree's boxes: box_expand(a, b).
static inline Box node_union(const Box& a, const Box& b) {
    return Box{V3{lib_min(a.mn.x, b.mn.x), lib_min(a.mn.y, b.mn.y), lib_min(a.mn.z, b.mn.z)},
               V3{lib_max(a.mx.x, b.mx.x), lib_max(a.mx.y, b.mx.y), lib_max(a.mx.z, b.mx.z)}};
}
// An SAH interior node's box over children l and r, with the operand order its trees have always had.
static inline Box sah_union(const Box& l, const Box& r) {
    return Box{V3{lib_min(r.mn.x, l.mn.x), lib_min(r.mn.y, l.mn.y), lib_min(r.mn.z, l.mn.z)},
               V3{lib_max(l.mx.x, r.mx.x), lib_max(r.mx.y, l.mx.y), lib_max(r.mx.z, l.mx.z)}};
}
// Stage (a).  With `sorted` the item order is already final (the device computed it) and only the shape and the boxes
// are built here; the shape depends on n alone.
struct Builder {
    const std::vector<Box>& boxes;
    std::vector<V3> centers;
    std::vector<int> order;
    std::vector<BuildNode> nodes;
    bool nan = false;
    bool sorted = false;
    const std::vector<uint8_t>* unbounded = nullptr;
    explicit Builder(const std::vector<Box>& b) : boxes(b) {
        order.resize(b.size());
        for (size_t i = 0; i < b.size(); ++i) order[i] = (int)i;
    }
    int build(int lo, int n, int depth) {
        if (!sorted) {
            if (centers.empty()) {
                centers.reserve(boxes.size());
                for (const Box& x : boxes) centers.push_back(box_center(x));
            }
            int axis = depth % 3;
            for (int i = lo; i < lo + n; ++i)
                if (std::isnan(comp(centers[order[i]], axis))) nan = true;  // bvh.rs:34 would panic
            std::stable_sort(order.begin() + lo, order.begin() + lo + n,
                             [&](int a, int b) { return comp(centers[a], axis) < comp(centers[b], axis); });
        }
        int id = (int)nodes.size();
        nodes.emplace_back();
        nodes[id].depth = depth;
        if (n == 1) {
            nodes[id].box = boxes[order[lo]];
            nodes[id].first = lo;
            nodes[id].count = 1;
            nodes[id].unbounded = unbounded && (*unbounded)[order[lo]];
        } else if (n == 2) {
            nodes[id].box = node_union(boxes[order[lo]], boxes[order[lo + 1]]);
            nodes[id].first = lo;
            nodes[id].count = 2;
            nodes[id].unbounded = unbounded && ((*unbounded)[order[lo]] || (*unbounded)[order[lo + 1]]);
        } else {
            int half = n / 2;
            int l = build(lo, half, depth + 1);
            int r = build(lo + half, n - half, depth + 1);
            nodes[id].left = l;
            nodes[id].right = r;
            nodes[id].box = node_union(nodes[l].box, nodes[r].box);
            nodes[id].unbounded = nodes[l].unbounded || nodes[r].unbounded;
        }
        return id;
    }
};
static inline float as_float(int i) {
    float f;
    memcpy(&f, &i, 4);
    return f;
}
constexpr int kSahMaxDepth = 22;   // binary levels below the root: keeps the traversal stack within FW_STACK
static double half_area(const Box& x) {
    double dx = (double)x.mx.x - x.mn.x, dy = (double)x.mx.y - x.mn.y, dz = (double)x.mx.z - x.mn.z;
    dx = std::max(dx, 0.0); dy = std::max(dy, 0.0); dz = std::max(dz, 0.0);
    return dx * dy + dy * dz + dz * dx;
}

// Stage (b) over `leaves` (node ids in DFS order); appends the interior to `nodes`, returns the root.  With `recs`
// (bvh_sah_device's records, `leaves` already in the device's final order) the splits are the device's and nothing is
// sorted here; either way the nodes are made by the same code below, so their boxes are bit for bit the same.
static int sah_tree(std::vector<BuildNode>& nodes, std::vector<int> leaves, const std::vector<SahRec>* recs) {
    nodes.reserve(nodes.size() + leaves.size());
    auto center = [&](int id, int a) {
        const Box& x = nodes[id].box;
        return a == 0 ? 0.5 * ((double)x.mn.x + x.mx.x) : a == 1 ? 0.5 * ((double)x.mn.y + x.mx.y) : 0.5 * ((double)x.mn.z + x.mx.z);
    };
    // Full-sweep SAH over the leaves, per node: order by centre along x, then (stably) y, then z; for every axis sweep
    // the split position.  All per-node state lives in slices [lo, lo + n) of buffers sized once (a node is done with
    // its slice before its children use theirs), and the leaf centres / areas are computed once: scene builds are on
    // the end-to-end path of every render (SURVEY §8 f3), and the per-node vectors + std::stable_sort's temporary
    // buffer were most of fw_scene_commit for a 500-object scene.
    const int nl = (int)leaves.size();
    const int n_bn = (int)nodes.size();
    std::vector<double> ctr[3];
    for (int a = 0; a < 3; ++a) {
        ctr[a].resize(n_bn);
        for (int id : leaves) {
            double c = center(id, a);
            ctr[a][id] = c == c ? c : INFINITY;   // NaN centre (unbounded box): any consistent place will do
        }
    }
    std::vector<int> ord[3];
    for (int a = 0; a < 3; ++a) ord[a].resize(nl);
    std::vector<double> right_area(nl);
    std::vector<int> merge_tmp(nl);
    auto sort_by = [&](int* v, int n, const std::vector<double>& key) {   // stable, ascending
        if (n <= 32) {
            for (int i = 1; i < n; ++i) {
                int x = v[i];
                double kx = key[x];
                int j = i;
                while (j > 0 && kx < key[v[j - 1]]) { v[j] = v[j - 1]; --j; }
                v[j] = x;
            }
            return;
        }
        // bottom-up merge sort over runs of 16 sorted by insertion
        for (int r = 0; r < n; r += 16) {
            int e = std::min(n, r + 16);
            for (int i = r + 1; i < e; ++i) {
                int x = v[i];
                double kx = key[x];
                int j = i;
                while (j > r && kx < key[v[j - 1]]) { v[j] = v[j - 1]; --j; }
                v[j] = x;
            }
        }
        int* src = v;
        int* dst = merge_tmp.data();
        for (int w = 16; w < n; w *= 2) {
            for (int r = 0; r < n; r += 2 * w) {
                int m = std::min(n, r + w), e = std::min(n, r + 2 * w);
                int i = r, j = m, o = r;
                while (i < m && j < e) dst[o++] = key[src[j]] < key[src[i]] ? src[j++] : src[i++];
                while (i < m) dst[o++] = src[i++];
                while (j < e) dst[o++] = src[j++];
            }
            std::swap(src, dst);
        }
        if (src != v) std::copy(src, src + n, v);
    };
    auto add_interior = [&](int l, int r, int depth) {
        int id = (int)nodes.size();
        nodes.emplace_back();
        nodes[id].depth = depth;
        nodes[id].left = l;
        nodes[id].right = r;
        nodes[id].box = sah_union(nodes[l].box, nodes[r].box);
        nodes[id].unbounded = nodes[l].unbounded || nodes[r].unbounded;
        return id;
    };
    std::function<int(int, int, int, int)> sah = [&](int lo, int n, int depth, int rec) -> int {
        if (n == 1) return leaves[lo];
        if (recs) {
            const SahRec& q = (*recs)[rec];
            int l = sah(lo, q.k, depth + 1, q.left);
            int r = sah(lo + q.k, n - q.k, depth + 1, q.right);
            return add_interior(l, r, depth);
        }
        int best_axis = -1, best_k = n / 2;
        double best_cost = INFINITY;
        int levels_needed = 0;
        while ((1 << levels_needed) < n) ++levels_needed;
        const bool balanced = depth + levels_needed >= kSahMaxDepth;
        int items_total = 0;
        for (int i = 0; i < n; ++i) items_total += nodes[leaves[lo + i]].count;
        for (int a = 0; a < 3; ++a) {
            int* tmp = ord[a].data() + lo;
            const int* from = a == 0 ? leaves.data() + lo : ord[a - 1].data() + lo;
            std::copy(from, from + n, tmp);
            sort_by(tmp, n, ctr[a]);
            Box acc = nodes[tmp[n - 1]].box;
            for (int i = n - 1; i > 0; --i) {
                acc = box_expand(acc, nodes[tmp[i]].box);
                right_area[lo + i] = half_area(acc);
            }
            acc = nodes[tmp[0]].box;
            int items_left = 0;
            for (int k = 1; k < n; ++k) {   // left = tmp[0..k), right = tmp[k..n)
                acc = box_expand(acc, nodes[tmp[k - 1]].box);
                items_left += nodes[tmp[k - 1]].count;
                if (balanced && k != n / 2) continue;
                double cost = half_area(acc) * items_left + right_area[lo + k] * (items_total - items_left);
                if (cost < best_cost) { best_cost = cost; best_axis = a; best_k = k; }
            }
        }
        if (best_axis < 0) { best_axis = 2; best_k = n / 2; }   // non-finite areas: any split is valid
        std::copy(ord[best_axis].begin() + lo, ord[best_axis].begin() + lo + n, leaves.begin() + lo);
        int l = sah(lo, best_k, depth + 1, -1);
        int r = sah(lo + best_k, n - best_k, depth + 1, -1);
        return add_interior(l, r, depth);
    };
    return sah(0, nl, 0, 0);
}

// Stage (b) on a device: the splits and the final leaf order come from bvh_sah_device.
static int sah_device(int device, std::vector<BuildNode>& nodes, const std::vector<int>& leaves, std::string& err) {
    std::vector<Box> boxes(leaves.size());
    std::vector<int> counts(leaves.size());
    for (size_t i = 0; i < leaves.size(); ++i) { boxes[i] = nodes[leaves[i]].box; counts[i] = nodes[leaves[i]].count; }
    std::vector<SahRec> recs;
    std::vector<int> leaf_order;
    if (!bvh_sah_device(device, boxes, counts, kSahMaxDepth, recs, leaf_order, err)) return -1;
    std::vector<int> ordered(leaves.size());
    for (size_t i = 0; i < leaves.size(); ++i) ordered[i] = leaves[leaf_order[i]];
    return sah_tree(nodes, std::move(ordered), &recs);
}

// Stage (c): collapse the binary tree two levels at a time into 4-wide nodes (breadth-first, so the top levels are
// contiguous).  A wide node holds the boxes of the binary node's grandchildren (or of a child that is itself a leaf).
// Skipping the intermediate child's box test cannot change which leaves are reached: the child's box contains the
// grandchild's, and the slab arithmetic (aabb.rs:38-47) is monotonic in the box planes, so "grandchild box hit" implies
// "child box hit" bit for bit.  The greedy collapse of an SAH interior reads structure, boxes and leaf codes only.
static void collapse(const std::vector<BuildNode>& nodes, int root, bool greedy, FlatBVH& out) {
    auto leaf_code = [](const BuildNode& n) { return ~(n.first * 2 + (n.count - 1)); };  // items [first, first+count)
    out.root_code = 0;
    struct Pending { int bn; int wide; int depth; };
    std::deque<Pending> q;
    q.push_back(Pending{root, 0, 1});
    int next_wide = 1;
    out.nodes.assign(8, float4{0, 0, 0, 0});
    while (!q.empty()) {
        Pending cur = q.front();
        q.pop_front();
        out.wide_depth = std::max(out.wide_depth, cur.depth);
        const BuildNode& n = nodes[cur.bn];
        int kids[4], nk = 0;
        if (greedy) {
            // greedy collapse: open the interior child with the largest box until the four slots are used
            kids[nk++] = n.left; kids[nk++] = n.right;
            while (nk < 4) {
                int pick = -1;
                double best = -1.0;
                for (int k = 0; k < nk; ++k)
                    if (nodes[kids[k]].count == 0) {
                        double a = half_area(nodes[kids[k]].box);
                        if (!(a <= best)) { best = a; pick = k; }
                    }
                if (pick < 0) break;
                int open = kids[pick];
                kids[pick] = nodes[open].left;
                kids[nk++] = nodes[open].right;
            }
        } else {
            for (int side : {n.left, n.right}) {
                const BuildNode& c = nodes[side];
                if (c.count > 0) kids[nk++] = side;
                else { kids[nk++] = c.left; kids[nk++] = c.right; }
            }
        }
        float lo[3][4], hi[3][4];
        int code[4], flag[4];
        for (int k = 0; k < 4; ++k) {
            if (k < nk) {
                const BuildNode& c = nodes[kids[k]];
                lo[0][k] = c.box.mn.x; lo[1][k] = c.box.mn.y; lo[2][k] = c.box.mn.z;
                hi[0][k] = c.box.mx.x; hi[1][k] = c.box.mx.y; hi[2][k] = c.box.mx.z;
                flag[k] = c.unbounded ? 1 : 0;
                if (c.count > 0) {
                    code[k] = leaf_code(c);
                } else {
                    code[k] = next_wide;
                    q.push_back(Pending{kids[k], next_wide, cur.depth + 1});
                    ++next_wide;
                    out.nodes.resize(8 * (size_t)next_wide, float4{0, 0, 0, 0});
                }
            } else {  // empty slot: an inverted box fails every slab test
                for (int a = 0; a < 3; ++a) { lo[a][k] = INFINITY; hi[a][k] = -INFINITY; }
                code[k] = (int)0x80000000;
                flag[k] = 0;
            }
        }
        float4* w = &out.nodes[8 * (size_t)cur.wide];
        for (int a = 0; a < 3; ++a) {
            w[a] = float4{lo[a][0], lo[a][1], lo[a][2], lo[a][3]};
            w[3 + a] = float4{hi[a][0], hi[a][1], hi[a][2], hi[a][3]};
        }
        w[6] = float4{as_float(code[0]), as_float(code[1]), as_float(code[2]), as_float(code[3])};
        w[7] = float4{as_float(flag[0]), as_float(flag[1]), as_float(flag[2]), as_float(flag[3])};
    }
}
}  // namespace

int build_bvh_on(int device, const std::vector<Box>& item_boxes, FlatBVH& out, std::string& err,
                 const std::vector<uint8_t>* item_unbounded) {
    out = FlatBVH();
    if (item_boxes.empty()) {
        err = "cannot build a BVH over zero items (the reference recurses forever: bvh.rs:59)";
        return FW_ERR_SCENE;
    }
    Builder b(item_boxes);
    b.unbounded = item_unbounded;
    if (device >= 0) {
        if (!bvh_leaf_order_device(device, item_boxes, b.order, b.nan, err)) return FW_ERR_CUDA;
        b.sorted = true;
    }
    if (!b.nan) {
        b.nodes.reserve(item_boxes.size() * 2);
        b.build(0, (int)item_boxes.size(), 0);
    }
    if (b.nan) {
        err = "Float comparison failed in BVH constructor (NaN centroid; bvh.rs:34)";
        return FW_ERR_SCENE;
    }
    const int median_root = 0;   // creation order: the root comes first
    out.items = b.order;
    for (const BuildNode& n : b.nodes) out.max_depth = std::max(out.max_depth, n.depth);
    out.root_box = b.nodes[median_root].box;
    if (b.nodes[median_root].count > 0) {
        out.root_code = ~(b.nodes[median_root].first * 2 + (b.nodes[median_root].count - 1));
        return FW_OK;
    }
    // Interior re-clustering.  Which items a ray tests is decided by the LEAF boxes alone: a leaf (bvh.rs Leaf /
    // DoubleLeaf, with the reference's box for it) is reached iff its own box test passes, because every ancestor's
    // box contains it and the slab arithmetic is monotonic in the box planes.  Any hierarchy that conservatively
    // bounds those leaves therefore yields the reference's candidate set, and the (t, DFS rank) merge rule does not
    // depend on visiting order.  The reference's tree (median split on a cycling axis) supplies the leaves, their
    // boxes and their DFS ranks; the interior nodes above them are rebuilt with a surface-area heuristic, which
    // roughly halves the boxes a ray has to test (FW_BVH_SAH=0 keeps the reference's interior).
    static const bool use_sah = [] { const char* e = getenv("FW_BVH_SAH"); return !e || atoi(e) != 0; }();
    int root = median_root;
    if (use_sah) {
        std::vector<int> leaves;
        for (int i = 0; i < (int)b.nodes.size(); ++i)
            if (b.nodes[i].count > 0) leaves.push_back(i);   // creation order == DFS order
        root = device >= 0 ? sah_device(device, b.nodes, leaves, err) : sah_tree(b.nodes, std::move(leaves), nullptr);
        if (root < 0) return FW_ERR_CUDA;
    }
    collapse(b.nodes, root, use_sah, out);
    return FW_OK;
}

static thread_local BvhDeviceScope* t_bvh_scope = nullptr;
BvhDeviceScope::BvhDeviceScope(int d) : device(d), prev(t_bvh_scope) { t_bvh_scope = this; }
BvhDeviceScope::~BvhDeviceScope() { t_bvh_scope = prev; }

__attribute__((noinline)) bool build_bvh(const std::vector<Box>& item_boxes, FlatBVH& out, std::string& err,
                                          const std::vector<uint8_t>* item_unbounded) {
    BvhDeviceScope* sc = t_bvh_scope;
    const int device = sc && sc->device >= 0 && item_boxes.size() >= kDeviceBvhMinItems ? sc->device : -1;
    const int rc = build_bvh_on(device, item_boxes, out, err, item_unbounded);
    if (rc != FW_OK && sc) sc->code = rc;
    return rc == FW_OK;
}

// ------------------------------------------------------------------------------------------------------
// Flattening
// ------------------------------------------------------------------------------------------------------
namespace {
struct M3 {
    V3 c[3];
};
static inline V3 mat_mul(const M3& m, V3 v) {  // ultraviolet Mat3 * Vec3
    return V3{m.c[0].x * v.x + m.c[1].x * v.y + m.c[2].x * v.z, m.c[0].y * v.x + m.c[1].y * v.y + m.c[2].y * v.z,
              m.c[0].z * v.x + m.c[1].z * v.y + m.c[2].z * v.z};
}
// ultraviolet Rotor3::into_matrix (see DESIGN.md "un-vendored arithmetic")
static M3 rotor_matrix(float s, float xy, float xz, float yz) {
    float s2 = s * s, bxy2 = xy * xy, bxz2 = xz * xz, byz2 = yz * yz;
    float s_bxy = s * xy, s_bxz = s * xz, s_byz = s * yz;
    float bxz_byz = xz * yz, bxy_byz = xy * yz, bxy_bxz = xy * xz;
    const float two = 2.0f;
    M3 m;
    m.c[0] = V3{s2 - bxy2 - bxz2 + byz2, -two * (bxz_byz + s_bxy), two * (bxy_byz - s_bxz)};
    m.c[1] = V3{two * (s_bxy - bxz_byz), s2 - bxy2 + bxz2 - byz2, -two * (s_byz + bxy_bxz)};
    m.c[2] = V3{two * (s_bxz + bxy_byz), two * (s_byz - bxy_bxz), s2 + bxy2 - bxz2 - byz2};
    return m;
}

// mesh.rs:221-242
static Box triangle_box(V3 p0, V3 p1, V3 p2) {
    Box b{vmin(p0, p1), vmax(p0, p1)};
    b.mn = vmin(b.mn, p2);
    b.mx = vmax(b.mx, p2);
    V3 size{fabsf(b.mx.x - b.mn.x), fabsf(b.mx.y - b.mn.y), fabsf(b.mx.z - b.mn.z)};
    if (size.x < 0.001f) { b.mn.x -= 0.001f; b.mx.x += 0.001f; }
    if (size.y < 0.001f) { b.mn.y -= 0.001f; b.mx.y += 0.001f; }
    if (size.z < 0.001f) { b.mn.z -= 0.001f; b.mx.z += 0.001f; }
    return b;
}
}  // namespace

// Rect3d helpers (see the device-record comment in flatten_scene).  `s` is the Rect3d's ShapeRec: faces are
// desc.shapes[s.i0 .. s.i0 + s.i1), each (min1, min2, max1, max2, k) with its plane in i0 & 3 (0 XY, 1 XZ, 2 YZ).
static bool rect3d_canonical(const SceneDesc& desc, const ShapeRec& s, float lo[3], float hi[3]) {
    auto bits_eq = [](float a, float b) { return memcmp(&a, &b, 4) == 0; };
    if (s.i1 != 6) return false;
    const ShapeRec* f = &desc.shapes[s.i0];
    static const int planes[6] = {0, 0, 1, 1, 2, 2};
    for (int k = 0; k < 6; ++k)
        if (f[k].kind != SH_RECT || (f[k].i0 & 3) != planes[k]) return false;
    lo[0] = f[0].f[0]; lo[1] = f[0].f[1]; hi[0] = f[0].f[2]; hi[1] = f[0].f[3]; hi[2] = f[0].f[4]; lo[2] = f[1].f[4];
    const float exp[6][5] = {{lo[0], lo[1], hi[0], hi[1], hi[2]}, {lo[0], lo[1], hi[0], hi[1], lo[2]},
                             {lo[0], lo[2], hi[0], hi[2], hi[1]}, {lo[0], lo[2], hi[0], hi[2], lo[1]},
                             {lo[1], lo[2], hi[1], hi[2], hi[0]}, {lo[1], lo[2], hi[1], hi[2], lo[0]}};
    for (int k = 0; k < 6; ++k)
        for (int c = 0; c < 5; ++c)
            if (!bits_eq(f[k].f[c], exp[k][c])) return false;
    return true;
}
static void rect3d_padded_box(const SceneDesc& desc, const ShapeRec& s, float lo[3], float hi[3]) {
    for (int a = 0; a < 3; ++a) { lo[a] = INFINITY; hi[a] = -INFINITY; }
    static const int A1[3] = {0, 0, 1}, A2[3] = {1, 2, 2}, AK[3] = {2, 1, 0};
    for (int f = 0; f < s.i1; ++f) {
        const ShapeRec& r = desc.shapes[s.i0 + f];
        int p = r.i0 & 3;
        lo[A1[p]] = fminf(lo[A1[p]], r.f[0]); hi[A1[p]] = fmaxf(hi[A1[p]], r.f[2]);
        lo[A2[p]] = fminf(lo[A2[p]], r.f[1]); hi[A2[p]] = fmaxf(hi[A2[p]], r.f[3]);
        lo[AK[p]] = fminf(lo[AK[p]], r.f[4]); hi[AK[p]] = fmaxf(hi[AK[p]], r.f[4]);
    }
    float ext = 0.0f;
    for (int a = 0; a < 3; ++a) ext = fmaxf(ext, fmaxf(fabsf(lo[a]), fabsf(hi[a])));
    float pad = 1e-3f * ext + 1e-4f;
    if (!(ext < INFINITY)) pad = 0.0f;  // no faces / non-finite: the inverted or infinite box decides
    for (int a = 0; a < 3; ++a) { lo[a] -= pad; hi[a] += pad; }
}

bool flatten_scene(const SceneDesc& desc, HostFlat& out, std::string& err) {
    out = HostFlat();
    if (desc.objects.empty()) {
        err = "No render objects added to scene! (scene.rs:161)";
        return false;
    }
    out.shapes = desc.shapes;
    out.mats = desc.mats;
    out.texs = desc.texs;
    // Rect3d device records.
    //  * canonical (the six faces Rect3d::new builds, rect3d.rs:18-80, all sharing lo / hi): f[0..5] = lo xyz, hi xyz
    //    exactly, f[7] = 1 — the kernels run the six face tests straight-line from those six numbers, without loading
    //    the face records;
    //  * anything else (a deserialised Rect3d may hold arbitrary faces): f[0..5] = a PADDED box around the union of
    //    the faces, f[7] = 0.  The kernels use it as a conservative pre-test before the face tests (rect3d.rs:89-100):
    //    a face can only be hit inside that box, and the padding (1e-3 of the extent + 1e-4) dwarfs every rounding
    //    difference between the slab arithmetic and the face test.
    // (pos / size themselves are only needed for the object's bounding box, computed below from desc.)
    for (ShapeRec& s : out.shapes) {
        if (s.kind != SH_RECT3D) continue;
        float lo[3], hi[3];
        if (rect3d_canonical(desc, s, lo, hi)) {
            for (int a = 0; a < 3; ++a) { s.f[a] = lo[a]; s.f[3 + a] = hi[a]; }
            s.f[6] = 0.0f; s.f[7] = 1.0f;
            continue;
        }
        rect3d_padded_box(desc, s, lo, hi);
        for (int a = 0; a < 3; ++a) { s.f[a] = lo[a]; s.f[3 + a] = hi[a]; }
        s.f[6] = 0.0f; s.f[7] = 0.0f;
    }
    {
        // uv is read only by ImageTexture::sample (texture.rs:296-309); checker forwards it to its children
        std::function<bool(int, int)> reads_uv = [&](int t, int depth) -> bool {
            if (t < 0 || t >= (int)desc.texs.size() || depth >= FW_MAX_TEXTURE_DEPTH) return false;
            const TexRec& r = desc.texs[t];
            if (r.kind == TEX_IMAGE) return true;
            if (r.kind == TEX_CHECKER) return reads_uv(r.a, depth + 1) || reads_uv(r.b, depth + 1);
            return false;
        };
        for (MatRec& m : out.mats) m.needs_uv = reads_uv(m.tex, 0) ? 1 : 0;
    }

    // Top-level tree occupies the front of nodes[]; it is appended after its size is known, so build
    // meshes into a side buffer first.
    std::vector<float4> mesh_nodes;
    int max_mesh_wide_depth = 0;
    std::vector<Box> mesh_root_box(desc.meshes.size());
    std::vector<int> mesh_node_root(desc.meshes.size());
    for (size_t mi = 0; mi < desc.meshes.size(); ++mi) {
        const MeshDesc& m = desc.meshes[mi];
        size_t ntri = m.indicies.size() / 3;
        std::vector<Box> tb(ntri);
        for (size_t t = 0; t < ntri; ++t)
            tb[t] = triangle_box(m.verts[m.indicies[3 * t]], m.verts[m.indicies[3 * t + 1]], m.verts[m.indicies[3 * t + 2]]);
        FlatBVH bvh;
        if (!build_bvh(tb, bvh, err)) return false;
        max_mesh_wide_depth = std::max(max_mesh_wide_depth, bvh.wide_depth);
        MeshRec rec;
        memset(&rec, 0, sizeof(rec));
        rec.root_code = bvh.root_code;  // tree-local; rebased below
        rec.tri_first = (int)(out.tri_verts.size() / 3);
        rec.tri_count = (int)ntri;
        rec.flags = (m.has_normals ? 1 : 0) | (m.has_uvs ? 2 : 0);
        rec.material = m.material;
        mesh_node_root[mi] = (int)(mesh_nodes.size() / 8);
        // child links are tree-local; rebased after the top-level tree's size is known
        mesh_nodes.insert(mesh_nodes.end(), bvh.nodes.begin(), bvh.nodes.end());
        mesh_root_box[mi] = bvh.root_box;
        rec.lo[0] = bvh.root_box.mn.x; rec.lo[1] = bvh.root_box.mn.y; rec.lo[2] = bvh.root_box.mn.z; rec.lo[3] = 0;
        rec.hi[0] = bvh.root_box.mx.x; rec.hi[1] = bvh.root_box.mx.y; rec.hi[2] = bvh.root_box.mx.z; rec.hi[3] = 0;
        for (size_t slot = 0; slot < ntri; ++slot) {
            int t = bvh.items[slot];
            uint32_t i0 = m.indicies[3 * t], i1 = m.indicies[3 * t + 1], i2 = m.indicies[3 * t + 2];
            V3 p0 = m.verts[i0], p1 = m.verts[i1], p2 = m.verts[i2];
            out.tri_verts.push_back(float4{p0.x, p0.y, p0.z, as_float(t)});
            out.tri_verts.push_back(float4{p1.x, p1.y, p1.z, 0});
            out.tri_verts.push_back(float4{p2.x, p2.y, p2.z, 0});
            if (m.has_normals) {
                V3 n0 = m.normals[i0], n1 = m.normals[i1], n2 = m.normals[i2];
                out.tri_normals.push_back(float4{n0.x, n0.y, n0.z, 0});
                out.tri_normals.push_back(float4{n1.x, n1.y, n1.z, 0});
                out.tri_normals.push_back(float4{n2.x, n2.y, n2.z, 0});
            } else {
                for (int k = 0; k < 3; ++k) out.tri_normals.push_back(float4{0, 0, 0, 0});
            }
            if (m.has_uvs) {
                out.tri_uvs.push_back(float2{m.uvs[2 * i0], m.uvs[2 * i0 + 1]});
                out.tri_uvs.push_back(float2{m.uvs[2 * i1], m.uvs[2 * i1 + 1]});
                out.tri_uvs.push_back(float2{m.uvs[2 * i2], m.uvs[2 * i2 + 1]});
            } else {  // mesh.rs:108
                out.tri_uvs.push_back(float2{0, 0});
                out.tri_uvs.push_back(float2{1, 0});
                out.tri_uvs.push_back(float2{0, 1});
            }
        }
        out.meshes.push_back(rec);
    }

    // shape bounding boxes (object space)
    std::function<bool(int, Box&)> shape_box = [&](int si, Box& b) -> bool {
        const ShapeRec& s = desc.shapes[si];
        switch (s.kind) {
            case SH_SPHERE: {  // sphere.rs:62-64
                float r = s.f[0];
                b = Box{V3{-1.0f * r, -1.0f * r, -1.0f * r}, V3{1.0f * r, 1.0f * r, 1.0f * r}};
                return true;
            }
            case SH_RECT: {  // rect.rs:75-86
                static const int A1[3] = {0, 0, 1}, A2[3] = {1, 2, 2}, AK[3] = {2, 1, 0};
                int p = s.i0 & 3;
                float lo[3] = {0, 0, 0}, hi[3] = {0, 0, 0};
                lo[A1[p]] = s.f[0]; lo[A2[p]] = s.f[1]; lo[AK[p]] = s.f[4] - 0.01f;
                hi[A1[p]] = s.f[2]; hi[A2[p]] = s.f[3]; hi[AK[p]] = s.f[4] + 0.01f;
                b = Box{V3{lo[0], lo[1], lo[2]}, V3{hi[0], hi[1], hi[2]}};
                return true;
            }
            case SH_RECT3D:  // rect3d.rs:102-104
                b = Box{V3{s.f[0], s.f[1], s.f[2]}, V3{s.f[0] + s.f[3], s.f[1] + s.f[4], s.f[2] + s.f[5]}};
                return true;
            case SH_MESH:
                b = mesh_root_box[s.i0];
                return true;
            case SH_DISK:  // disk.rs:85-90 (degenerate box preserved)
                b = Box{V3{-s.f[0], 0.0f, s.f[0]}, V3{-s.f[0], 0.001f, s.f[0]}};
                return true;
            case SH_CYLINDER:  // cylinder.rs:92-97
            case SH_CONE:      // cone.rs:90-95
                b = Box{V3{-s.f[0], 0.0f, -s.f[0]}, V3{s.f[0], s.f[1], s.f[0]}};
                return true;
            case SH_MEDIUM:  // volume.rs:84-86
                return shape_box(s.i0, b);
        }
        err = "bad shape kind";
        return false;
    };

    // Does the shape's bounding box really bound its geometry?  Disk's does not (disk.rs:85-90 is degenerate in
    // x and z); a deserialised Rect3d may list faces outside pos..pos+size.
    std::function<bool(int)> shape_unbounded = [&](int si) -> bool {
        const ShapeRec& s = desc.shapes[si];
        if (s.kind == SH_DISK) return true;
        if (s.kind == SH_MEDIUM) return shape_unbounded(s.i0);
        if (s.kind == SH_RECT3D) {
            Box b;
            shape_box(si, b);
            for (int f = 0; f < s.i1; ++f) {
                Box fb;
                shape_box(s.i0 + f, fb);
                if (fb.mn.x < b.mn.x - 0.011f || fb.mn.y < b.mn.y - 0.011f || fb.mn.z < b.mn.z - 0.011f ||
                    fb.mx.x > b.mx.x + 0.011f || fb.mx.y > b.mx.y + 0.011f || fb.mx.z > b.mx.z + 0.011f)
                    return true;
            }
        }
        return false;
    };
    std::vector<uint8_t> obj_unbounded(desc.objects.size(), 0);

    size_t nobj = desc.objects.size();
    out.obj_aabb.resize(nobj);
    int mesh_ordinal = 0;
    for (size_t i = 0; i < nobj; ++i) {
        const ObjectDesc& o = desc.objects[i];
        const ShapeRec& s = desc.shapes[o.shape];
        M3 R = rotor_matrix(o.rotor[0], o.rotor[1], o.rotor[2], o.rotor[3]);       // scene.rs:284
        M3 Ri = rotor_matrix(o.rotor[0], -o.rotor[1], -o.rotor[2], -o.rotor[3]);   // scene.rs:285 (reversed)
        float trace = R.c[0].x + R.c[1].y + R.c[2].z;
        float cos_trace = 0.5f * (trace - 1.0f);
        bool rotated = cos_trace < 0.999f;
        Box bbox;
        if (!shape_box(o.shape, bbox)) return false;
        Box rb;
        if (rotated) {  // scene.rs:186-208
            V3 mn{10e9f * 1.0f, 10e9f * 1.0f, 10e9f * 1.0f};
            V3 mx{-10e9f * 1.0f, -10e9f * 1.0f, -10e9f * 1.0f};
            for (int a = 0; a < 2; ++a)
                for (int bq = 0; bq < 2; ++bq)
                    for (int c = 0; c < 2; ++c) {
                        V3 corner{a == 0 ? bbox.mn.x : bbox.mx.x, bq == 0 ? bbox.mn.y : bbox.mx.y, c == 0 ? bbox.mn.z : bbox.mx.z};
                        V3 np = mat_mul(R, corner);
                        mx = V3{fmaxf(np.x, mx.x), fmaxf(np.y, mx.y), fmaxf(np.z, mx.z)};
                        mn = V3{fminf(np.x, mn.x), fminf(np.y, mn.y), fminf(np.z, mn.z)};
                    }
            rb = Box{mn, mx};
        } else {
            rb = bbox;
        }
        out.obj_aabb[i] = Box{V3{rb.mn.x + o.position.x, rb.mn.y + o.position.y, rb.mn.z + o.position.z},
                              V3{rb.mx.x + o.position.x, rb.mx.y + o.position.y, rb.mx.z + o.position.z}};
        int flags = s.kind | (rotated ? OBJ_ROTATED : 0) | (o.flip_normals ? OBJ_FLIP : 0);
        if (s.kind == SH_MESH) {   // ordinal among the top-level meshes (scene order); only meaningful when there are <= 8
            flags |= (mesh_ordinal & (FW_MAX_WALK_MESHES - 1)) << OBJ_MESH_ORD_SHIFT;
            ++mesh_ordinal;
        }
        out.obj_posr.push_back(float4{o.position.x, o.position.y, o.position.z, s.kind == SH_SPHERE ? s.f[0] : 0.0f});
        out.obj_meta.push_back(int4{flags, s.material, o.shape, 0});
        for (int c = 0; c < 3; ++c) {
            out.obj_rot.push_back(float4{R.c[c].x, R.c[c].y, R.c[c].z, 0});
            out.obj_irot.push_back(float4{Ri.c[c].x, Ri.c[c].y, Ri.c[c].z, 0});
        }
        if (s.kind == SH_MEDIUM) out.has_medium = true;
        if (s.kind == SH_MESH) out.has_mesh = out.has_top_mesh = true;
        if (s.kind == SH_MEDIUM && desc.shapes[s.i0].kind == SH_MESH) out.has_mesh = out.has_medium_mesh = true;
        obj_unbounded[i] = shape_unbounded(o.shape) ? 1 : 0;
        if (obj_unbounded[i]) out.has_unbounded = true;
    }

    // linear-scan program (fw_types.h LinItem): the objects in scene order (scene.rs:137-149)
    {
        std::vector<float4>& W = out.lin_words;
        bool world = true;            // the kernel starts in world space (position +0, unrotated)
        int space_obj = -1;           // object whose transform defines the current space (when !world)
        bool space_has_rects = false; // the current space's XFORM item carries LIN_SPACE_HAS_RECTS
        size_t xform_word = 0;        // index of the current space's XFORM item
        auto bits_eq = [](float a, float b) { return memcmp(&a, &b, 4) == 0; };
        auto is_pzero = [](float a) { uint32_t u; memcpy(&u, &a, 4); return u == 0u; };  // +0.0 only: x - (+0) == x exactly
        for (size_t i = 0; i < nobj; ++i) {
            const ObjectDesc& o = desc.objects[i];
            const ShapeRec& s = out.shapes[o.shape];  // device copy: Rect3d carries its padded face box
            bool rotated = (out.obj_meta[i].x & OBJ_ROTATED) != 0;
            bool simple = s.kind == SH_RECT || s.kind == SH_RECT3D || s.kind == SH_SPHERE;
            if (!simple) {
                out.lin_generic = true;
                W.push_back(float4{0, as_float(LIN_GENERIC), as_float((int)i), 0});
                continue;
            }
            // ray -> object space (scene.rs:242-253), shared with the previous object when the transform is the same
            bool want_world = !rotated && is_pzero(o.position.x) && is_pzero(o.position.y) && is_pzero(o.position.z);
            bool same = false;
            if (want_world) same = world;
            else if (!world && space_obj >= 0 && !rotated && !(out.obj_meta[space_obj].x & OBJ_ROTATED)) {
                const ObjectDesc& q = desc.objects[space_obj];
                same = bits_eq(q.position.x, o.position.x) && bits_eq(q.position.y, o.position.y) && bits_eq(q.position.z, o.position.z);
            }
            const bool rects = s.kind != SH_SPHERE;
            // the kernel starts in world space WITHOUT the shared-division state: a space whose first rectangle
            // arrives later (or the initial world space) gets an XFORM item that sets it up
            if (!same || (rects && !space_has_rects)) {
                xform_word = W.size();
                W.push_back(float4{o.position.x, as_float(rotated ? LIN_XFORM_R : LIN_XFORM_T), o.position.y, o.position.z});
                if (rotated) for (int c = 0; c < 3; ++c) W.push_back(out.obj_irot[3 * i + c]);
                world = want_world;
                space_obj = (int)i;
                space_has_rects = false;
            }
            if (rects && !space_has_rects) {
                int tpw;
                memcpy(&tpw, &W[xform_word].y, 4);
                W[xform_word].y = as_float(tpw | LIN_SPACE_HAS_RECTS);
                space_has_rects = true;
            }
            if (s.kind == SH_SPHERE) {
                W.push_back(float4{s.f[0], as_float(LIN_SPHERE), as_float((int)i), 0});
            } else if (s.kind == SH_RECT) {
                out.lin_rect_tests += 1;
                W.push_back(float4{s.f[4], as_float(LIN_RECT | ((s.i0 & 3) << 8)), as_float((int)i), as_float(0)});
                W.push_back(float4{s.f[0], s.f[1], s.f[2], s.f[3]});
            } else {
                // Rect3d: the six canonical faces of Rect3d::new (rect3d.rs:18-80) collapse into one BOX6 item
                const ShapeRec* f = &desc.shapes[s.i0];
                float lo[3], hi[3];
                out.lin_rect_tests += s.i1;
                if (rect3d_canonical(desc, desc.shapes[o.shape], lo, hi)) {
                    float plo[3], phi[3];
                    rect3d_padded_box(desc, desc.shapes[o.shape], plo, phi);
                    W.push_back(float4{lo[0], as_float(LIN_BOX6), as_float((int)i), lo[1]});
                    W.push_back(float4{lo[2], hi[0], hi[1], hi[2]});
                    W.push_back(float4{plo[0], plo[1], plo[2], phi[0]});
                    W.push_back(float4{phi[1], phi[2], 0, 0});
                } else {
                    for (int k = 0; k < s.i1; ++k) {
                        W.push_back(float4{f[k].f[4], as_float(LIN_RECT | ((f[k].i0 & 3) << 8)), as_float((int)i), as_float(k)});
                        W.push_back(float4{f[k].f[0], f[k].f[1], f[k].f[2], f[k].f[3]});
                    }
                }
            }
        }
        W.push_back(float4{0, as_float(LIN_END), 0, 0});
    }

    // Triangle vertices pre-permuted for the three possible dominant axes of a ray (mesh.rs:146-153 permutes every vertex
    // per test: nine selects the mesh walk's test phase does not have to execute; same values, so the same bits).
    {
        const size_t nt = out.tri_verts.size() / 3;
        out.tri_perm.resize(out.tri_verts.size() * 3);
        for (int kz = 0; kz < 3; ++kz) {
            const int kx = (kz + 1) % 3, ky = (kx + 1) % 3;
            for (size_t i = 0; i < nt * 3; ++i) {
                const float4& v = out.tri_verts[i];
                const float c[3] = {v.x, v.y, v.z};
                out.tri_perm[(size_t)kz * nt * 3 + i] = float4{c[kx], c[ky], c[kz], v.w};
            }
        }
    }

    // top-level BVH (bvh.rs:79-98), always built: linear-scan renders simply do not use it
    FlatBVH top;
    if (!build_bvh(out.obj_aabb, top, err, &obj_unbounded)) return false;
    // traversal stack: up to 3 deferred siblings per wide level, on both levels, plus EXIT / ENTER markers
    if (3 * (top.wide_depth + max_mesh_wide_depth) + 8 > 96) {   // FW_STACK (intersect.cuh)
        err = "BVH deeper than the traversal stack";
        return false;
    }
    out.top_items = top.items;
    {
        // The top-level tree's leaves with the reference's boxes for them, in DFS order: small scenes scan this list
        // straight through instead of walking the tree (kernels_extend.cu extend_pass1_small_kernel).
        std::vector<std::pair<int, std::pair<float4, float4>>> leaves;
        auto add_leaf = [&](int code, const float* lo, const float* hi) {
            const int packed = ~code, first = packed >> 1, count = (packed & 1) + 1;
            leaves.push_back({first, {float4{lo[0], lo[1], lo[2], as_float(first)}, float4{hi[0], hi[1], hi[2], as_float(count)}}});
        };
        if (top.root_code < 0) {
            const float lo[3] = {top.root_box.mn.x, top.root_box.mn.y, top.root_box.mn.z}, hi[3] = {top.root_box.mx.x, top.root_box.mx.y, top.root_box.mx.z};
            add_leaf(top.root_code, lo, hi);
        }
        for (size_t n = 0; n + 7 < top.nodes.size(); n += 8) {
            const float4* q = &top.nodes[n];
            const float* rows[6] = {&q[0].x, &q[1].x, &q[2].x, &q[3].x, &q[4].x, &q[5].x};
            int codes[4];
            memcpy(codes, &q[6], 16);
            for (int k = 0; k < 4; ++k) {
                if (codes[k] >= 0 || codes[k] == (int)0x80000000) continue;
                const float lo[3] = {rows[0][k], rows[1][k], rows[2][k]}, hi[3] = {rows[3][k], rows[4][k], rows[5][k]};
                add_leaf(codes[k], lo, hi);
            }
        }
        std::sort(leaves.begin(), leaves.end(), [](const auto& a, const auto& b) { return a.first < b.first; });
        for (const auto& l : leaves) { out.top_leaves.push_back(l.second.first); out.top_leaves.push_back(l.second.second); }
    }
    for (int obj : top.items) {
        out.leaf_posr.push_back(out.obj_posr[obj]);
        int4 m = out.obj_meta[obj];
        m.w = obj;
        out.leaf_meta.push_back(m);
    }
    {
        out.top_wide_depth = top.wide_depth;
        out.mesh_wide_depth = max_mesh_wide_depth;
        int max_prim = 0;
        bool roots_wide = top.root_code >= 0;
        for (const ObjectDesc& o : desc.objects) {
            const ShapeRec& sh = desc.shapes[o.shape];
            if (sh.kind == SH_MESH) {
                out.n_top_meshes++;
                max_prim = std::max(max_prim, out.meshes[sh.i0].tri_count - 1);
                roots_wide = roots_wide && out.meshes[sh.i0].root_code >= 0;
            } else if (sh.kind == SH_RECT3D) {
                max_prim = std::max(max_prim, sh.i1 - 1);
            }
        }
        if (out.n_top_meshes <= FW_MAX_WALK_MESHES)
            for (size_t rank = 0; rank < top.items.size(); ++rank) {
                const int4& m = out.obj_meta[top.items[rank]];
                if ((m.x & OBJ_KIND_MASK) == SH_MESH) out.mesh_rank[(m.x >> OBJ_MESH_ORD_SHIFT) & (FW_MAX_WALK_MESHES - 1)] = (int)rank;
            }
        int rank_bits = 1;
        while (rank_bits < 31 && ((size_t)1 << rank_bits) < desc.objects.size()) ++rank_bits;
        out.walk_prim_bits = 32 - rank_bits;
        const bool key_fits = (size_t)max_prim < ((size_t)1 << out.walk_prim_bits) && ((size_t)1 << rank_bits) >= desc.objects.size();
        out.walk_ok = roots_wide && key_fits && out.n_top_meshes >= 1 && out.n_top_meshes <= FW_MAX_WALK_MESHES && 3 * top.wide_depth + 4 <= 64 &&
                      3 * max_mesh_wide_depth + 4 <= 64;
    }
    out.top_depth = top.max_depth;
    out.top_nodes = (int)(top.nodes.size() / 8);
    out.nodes = top.nodes;
    out.top_root_box = top.root_box;
    out.top_root_code = top.root_code;
    // A ray with an all-NaN direction (e.g. after scattering off a zero-length interpolated normal) passes every
    // slab test (f32::max/min ignore NaN, aabb.rs:46-48) and is then "hit" by every primitive whose rejection
    // tests are all comparisons (NaN compares false): AARect (rect.rs:51,55), Triangle (mesh.rs:170-186), Disk,
    // Cone; Sphere, Cylinder and ConstantMedium reject it (their accept test is a comparison).  bvh.rs:128,141
    // (`left.t < right.t` false -> right) and scene.rs:142 (NaN `closest` never rejects) both make the LAST
    // accepting item win, so the answer does not depend on the ray and is precomputed here; the kernels return it
    // directly instead of walking the entire tree (milliseconds for one path).
    {
        auto accepts = [&](int obj, int& prim) -> bool {
            const ShapeRec& sh = desc.shapes[desc.objects[obj].shape];
            prim = 0;
            switch (sh.kind) {
                case SH_RECT: case SH_DISK: case SH_CONE: return true;
                case SH_RECT3D: prim = sh.i1 - 1; return sh.i1 > 0;
                case SH_MESH: prim = out.meshes[sh.i0].tri_count - 1; return true;   // last triangle slot
                default: return false;
            }
        };
        for (int rank = (int)out.top_items.size() - 1; rank >= 0; --rank) {
            int prim;
            if (accepts(out.top_items[rank], prim)) { out.nan_bvh_obj = out.top_items[rank]; out.nan_bvh_prim = prim; break; }
        }
        for (int obj = (int)desc.objects.size() - 1; obj >= 0; --obj) {
            int prim;
            if (accepts(obj, prim)) { out.nan_lin_obj = obj; out.nan_lin_prim = prim; break; }
        }
    }
    // append the mesh trees, rebasing child links and roots
    int base = (int)(out.nodes.size() / 8);
    size_t start = out.nodes.size();
    out.nodes.insert(out.nodes.end(), mesh_nodes.begin(), mesh_nodes.end());
    for (size_t mi = 0; mi < out.meshes.size(); ++mi) {
        int tree_off = mesh_node_root[mi];
        int tree_end = (mi + 1 < out.meshes.size()) ? mesh_node_root[mi + 1] : (int)(mesh_nodes.size() / 8);
        for (int n = tree_off; n < tree_end; ++n) {
            float4& codes = out.nodes[start + 8 * (size_t)n + 6];
            float* cf = &codes.x;
            for (int k = 0; k < 4; ++k) {
                int a;
                memcpy(&a, &cf[k], 4);
                if (a >= 0) {
                    a += base + tree_off;
                    cf[k] = as_float(a);
                }
            }
        }
        if (out.meshes[mi].root_code >= 0) out.meshes[mi].root_code += base + tree_off;
    }
    return true;
}

// camera.rs:74-107
CameraRec make_camera(const RenderParamsHost& p) {
    const float PI_F = 3.14159265358979323846f;
    auto sub = [](V3 a, V3 b) { return V3{a.x - b.x, a.y - b.y, a.z - b.z}; };
    auto mulf = [](float s, V3 a) { return V3{s * a.x, s * a.y, s * a.z}; };
    auto cross = [](V3 a, V3 b) { return V3{a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x}; };
    auto norm = [](V3 a) {
        float m = sqrtf((a.x * a.x) + (a.y * a.y) + (a.z * a.z));
        return V3{a.x / m, a.y / m, a.z / m};
    };
    V3 cam_pos{p.cam_pos[0], p.cam_pos[1], p.cam_pos[2]}, look_at{p.look_at[0], p.look_at[1], p.look_at[2]};
    float theta = p.vfov * PI_F / 180.0f;
    V3 w = norm(sub(cam_pos, look_at));
    V3 u = norm(cross(V3{0, 1, 0}, w));
    V3 v = cross(w, u);
    float half_height = tanf(theta / 2.0f);
    float half_width = half_height * (float)p.width / (float)p.height;
    V3 ll = sub(sub(sub(cam_pos, mulf(half_width * p.focus_dist, u)), mulf(half_height * p.focus_dist, v)),
                V3{w.x * p.focus_dist, w.y * p.focus_dist, w.z * p.focus_dist});
    V3 hor = mulf(2.0f * half_width * p.focus_dist, u);
    V3 ver = mulf(2.0f * half_height * p.focus_dist, v);
    CameraRec c;
    auto put = [](float* d, V3 s) { d[0] = s.x; d[1] = s.y; d[2] = s.z; };
    put(c.position, cam_pos); put(c.horizontal, hor); put(c.vertical, ver); put(c.lower_left, ll);
    put(c.u, u); put(c.v, v); put(c.w, w);
    c.lens_radius = p.aperture / 2.0f;
    return c;
}

}  // namespace fw
