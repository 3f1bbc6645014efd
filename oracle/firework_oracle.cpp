// firework_oracle.cpp — CPU ORACLE (TEST INFRASTRUCTURE, NOT PRODUCT CODE).
//
// A C++ restatement of the rendering hot path of ritobanrc/firework, written by reading the Rust
// sources and re-expressing each function with the same operation order in IEEE f32.  Every function
// cites the reference file:line it follows (paths relative to /root/reference).
//
// Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may load
// this library.  The product (firework_b200/) never links, imports or calls it.
//
// PARITY: the reference has no tests, no golden vectors, and cannot be compiled here (no Rust toolchain, nightly
// features, un-vendored crates), so no function of this restatement is pinned by a reference TEST.  What pins it
// is the reference's committed ARTEFACTS (fixtures + generating scripts under tests/golden/):
//   * suzanne.png / teapot.png / conics.png (renders of the committed scenes/*.yml with the examples' cameras),
//     cornell_box.png and Earth.png (deterministic example scenes): this oracle and the CUDA path reproduce them end
//     to end (8x8 box means: oracle ~35 dB at 24 spp, noise-limited; GPU 43-51 dB at 256-1000 spp) — geometry,
//     orientation, every shape's hit routine, normals, image-texture uv, sky, lights, output transform;
//   * cornell_box.png patch means (handedness, rotation sign, radiometry of the path loop);
//   * the Rotor3 values and mesh arrays serialised in scenes/suzanne.yml / teapot.yml (rotor constructors, OBJ ingestion).
// Everything else (per-function operation order, tie rules, quirks) is a reading of the cited lines, checked by
// self-consistency tests (tests/test_oracle.py): PARITY UNPINNED at that granularity.
// Arithmetic that lives in un-vendored crates is restated from their published algorithms:
//   ultraviolet 0.5.1 (Vec3/Mat3/Rotor3; Cargo.lock:1001)  — plain component f32 arithmetic, dot/cross
//       without fused multiply-add, normalized() = component / mag()   [unverifiable here]
//   tiny-rng 0.1.0 (LcRng; Cargo.lock:965) — NOT restated.  The sequential per-pixel LCG stream is
//       replaced, in the oracle and in the CUDA path alike, by a counter-based Philox4x32-10 keyed
//       by (seed; pixel, sample, bounce, stream-kind, block).  See DESIGN.md "RNG".
//
// Build: oracle/Makefile  (parity build: -O2 -ffp-contract=off; timing build: -O3 -march=native,
// still -ffp-contract=off so that both builds give identical bits).

#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <memory>
#include <string>
#include <vector>
#ifdef _OPENMP
#include <omp.h>
#endif

namespace orc {

// ------------------------------------------------------------------------------------------------
// ultraviolet::Vec3 / Vec2 / Mat3 (scalar f32), restated.
// ------------------------------------------------------------------------------------------------
struct Vec2 {
    float x, y;
};
struct Vec3 {
    float x, y, z;
    float operator[](int i) const { return i == 0 ? x : (i == 1 ? y : z); }
    float& at(int i) { return i == 0 ? x : (i == 1 ? y : z); }
};
static inline Vec3 v3(float x, float y, float z) { return Vec3{x, y, z}; }
static inline Vec3 operator+(Vec3 a, Vec3 b) { return v3(a.x + b.x, a.y + b.y, a.z + b.z); }
static inline Vec3 operator-(Vec3 a, Vec3 b) { return v3(a.x - b.x, a.y - b.y, a.z - b.z); }
static inline Vec3 operator-(Vec3 a) { return v3(-a.x, -a.y, -a.z); }
static inline Vec3 operator*(Vec3 a, Vec3 b) { return v3(a.x * b.x, a.y * b.y, a.z * b.z); }
static inline Vec3 operator*(float s, Vec3 a) { return v3(s * a.x, s * a.y, s * a.z); }
static inline Vec3 operator*(Vec3 a, float s) { return v3(a.x * s, a.y * s, a.z * s); }
static inline Vec3 operator/(Vec3 a, float s) { return v3(a.x / s, a.y / s, a.z / s); }
static inline float dot(Vec3 a, Vec3 b) { return (a.x * b.x) + (a.y * b.y) + (a.z * b.z); }
static inline float mag_sq(Vec3 a) { return (a.x * a.x) + (a.y * a.y) + (a.z * a.z); }
static inline float mag(Vec3 a) { return std::sqrt(mag_sq(a)); }
static inline Vec3 cross(Vec3 a, Vec3 b) {
    return v3(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x);
}
static inline Vec3 normalized(Vec3 a) {
    float m = mag(a);
    return v3(a.x / m, a.y / m, a.z / m);
}
// f32::max / f32::min: NaN-ignoring (== fmaxf / fminf).
static inline float fmax_(float a, float b) { return std::fmax(a, b); }
static inline float fmin_(float a, float b) { return std::fmin(a, b); }
static inline Vec3 min_by_component(Vec3 a, Vec3 b) {
    return v3(fmin_(a.x, b.x), fmin_(a.y, b.y), fmin_(a.z, b.z));
}
static inline Vec3 max_by_component(Vec3 a, Vec3 b) {
    return v3(fmax_(a.x, b.x), fmax_(a.y, b.y), fmax_(a.z, b.z));
}
static inline Vec2 operator*(float s, Vec2 a) { return Vec2{s * a.x, s * a.y}; }
static inline Vec2 operator+(Vec2 a, Vec2 b) { return Vec2{a.x + b.x, a.y + b.y}; }

// Mat3: column-major, `m[i][j]` = column i, row j (ultraviolet Mat3 { cols: [Vec3; 3] }).
struct Mat3 {
    Vec3 cols[3];
};
static inline Vec3 operator*(const Mat3& m, Vec3 v) {
    const Vec3 &a = m.cols[0], &b = m.cols[1], &c = m.cols[2];
    return v3(a.x * v.x + b.x * v.y + c.x * v.z, a.y * v.x + b.y * v.y + c.y * v.z,
              a.z * v.x + b.z * v.y + c.z * v.z);
}
// ultraviolet Rotor3 {s, bv{xy,xz,yz}}::into_matrix (restated from the published formula; the sign
// convention is checked against cornell_box.png and the from_rotation_xz values in scenes/*.yml).
struct Rotor3 {
    float s, xy, xz, yz;
};
static Mat3 rotor_into_matrix(Rotor3 r) {
    float s2 = r.s * r.s;
    float bxy2 = r.xy * r.xy, bxz2 = r.xz * r.xz, byz2 = r.yz * r.yz;
    float s_bxy = r.s * r.xy, s_bxz = r.s * r.xz, s_byz = r.s * r.yz;
    float bxz_byz = r.xz * r.yz, bxy_byz = r.xy * r.yz, bxy_bxz = r.xy * r.xz;
    const float two = 2.0f;
    Mat3 m;
    m.cols[0] = v3(s2 - bxy2 - bxz2 + byz2, -two * (bxz_byz + s_bxy), two * (bxy_byz - s_bxz));
    m.cols[1] = v3(two * (s_bxy - bxz_byz), s2 - bxy2 + bxz2 - byz2, -two * (s_byz + bxy_bxz));
    m.cols[2] = v3(two * (s_bxz + bxy_byz), two * (s_byz - bxy_bxz), s2 + bxy2 - bxz2 - byz2);
    return m;
}
static Rotor3 rotor_reversed(Rotor3 r) { return Rotor3{r.s, -r.xy, -r.xz, -r.yz}; }

// Rust `as usize` / `as u32` / `as u8` from f32: saturating, NaN -> 0.
static inline uint64_t f32_as_usize(float f) {
    if (!(f == f)) return 0;
    if (f <= 0.0f) return 0;
    if (f >= 18446744073709551616.0f) return UINT64_MAX;
    return (uint64_t)f;
}
static inline uint32_t f32_as_u32(float f) {
    if (!(f == f)) return 0;
    if (f <= 0.0f) return 0;
    if (f >= 4294967296.0f) return UINT32_MAX;
    return (uint32_t)f;
}
static inline uint8_t f32_as_u8(float f) {
    if (!(f == f)) return 0;
    if (f <= 0.0f) return 0;
    if (f >= 255.0f) return 255;
    return (uint8_t)f;
}

static const float PI_F = 3.14159265358979323846f;

// ------------------------------------------------------------------------------------------------
// RNG: Philox4x32-10, counter = (block, bounce<<8 | kind, sample, pixel), key = (seed_lo, seed_hi).
// Replaces tiny_rng::LcRng (see header).  rand_f32 = (u32 >> 8) * 2^-24  in [0, 1).
// ------------------------------------------------------------------------------------------------
enum StreamKind : uint32_t { STREAM_CAMERA = 0, STREAM_SCATTER = 1, STREAM_MEDIUM = 2 };

static inline void philox4x32_10(const uint32_t ctr_in[4], const uint32_t key_in[2], uint32_t out[4]) {
    uint32_t c0 = ctr_in[0], c1 = ctr_in[1], c2 = ctr_in[2], c3 = ctr_in[3];
    uint32_t k0 = key_in[0], k1 = key_in[1];
    for (int r = 0; r < 10; ++r) {
        uint64_t p0 = (uint64_t)0xD2511F53u * c0;
        uint64_t p1 = (uint64_t)0xCD9E8D57u * c2;
        uint32_t hi0 = (uint32_t)(p0 >> 32), lo0 = (uint32_t)p0;
        uint32_t hi1 = (uint32_t)(p1 >> 32), lo1 = (uint32_t)p1;
        uint32_t n0 = hi1 ^ c1 ^ k0;
        uint32_t n1 = lo1;
        uint32_t n2 = hi0 ^ c3 ^ k1;
        uint32_t n3 = lo0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}
static inline float u32_to_unit_f32(uint32_t x) { return (float)(x >> 8) * (1.0f / 16777216.0f); }

struct Rng {
    // keyed mode
    uint32_t key[2] = {0, 0};
    uint32_t pixel = 0, sample = 0, bounce = 0, kind = 0;
    uint32_t idx = 0;
    uint32_t buf[4];
    // array mode (explicit uniforms for the scatter-step gate)
    const float* arr = nullptr;
    int arr_n = 0, arr_i = 0;
    int arr_overrun = 0;

    void seed(uint64_t s) { key[0] = (uint32_t)s; key[1] = (uint32_t)(s >> 32); }
    void begin(uint32_t px, uint32_t smp) { pixel = px; sample = smp; }
    void set_stream(uint32_t b, uint32_t k) { bounce = b; kind = k; idx = 0; }
    float rand_f32() {
        if (arr) {
            if (arr_i >= arr_n) { arr_overrun = 1; return 0.5f; }
            return arr[arr_i++];
        }
        uint32_t lane = idx & 3u;
        if (lane == 0) {
            uint32_t ctr[4] = {idx >> 2, (bounce << 8) | kind, sample, pixel};
            philox4x32_10(ctr, key, buf);
        }
        ++idx;
        return u32_to_unit_f32(buf[lane]);
    }
    // One draw keyed by an object id, independent of traversal order (ConstantMedium, volume.rs:67).
    float rand_keyed(uint32_t id) {
        if (arr) return rand_f32();
        uint32_t ctr[4] = {id, (bounce << 8) | (uint32_t)STREAM_MEDIUM, sample, pixel};
        uint32_t o[4];
        philox4x32_10(ctr, key, o);
        return u32_to_unit_f32(o[0]);
    }
};

// ------------------------------------------------------------------------------------------------
// Counters (instrumentation only; per-thread, summed by the caller).
// ------------------------------------------------------------------------------------------------
struct Counters {
    uint64_t rays = 0, aabb_tests = 0, prim_tests = 0;
    // per-kind breakdown of prim_tests + object transforms, for the roofline's algorithmic flop / byte counts
    uint64_t sphere = 0, rect = 0, tri = 0, conic = 0, xform_rot = 0, xform_trans = 0;
};
static thread_local Counters g_cnt;

// ------------------------------------------------------------------------------------------------
// ray.rs:5-30
// ------------------------------------------------------------------------------------------------
struct Ray {
    Vec3 origin, dir;
    Vec3 point(float t) const { return origin + t * dir; }  // ray.rs:27-29
};

// ------------------------------------------------------------------------------------------------
// aabb.rs
// ------------------------------------------------------------------------------------------------
struct AABB {
    Vec3 min, max;
    static AABB from_two_points(Vec3 p0, Vec3 p1) {  // aabb.rs:23-28
        return AABB{min_by_component(p0, p1), max_by_component(p0, p1)};
    }
    bool hit(const Ray& ray, float tmin, float tmax) const {  // aabb.rs:30-50
        ++g_cnt.aabb_tests;
        for (int a = 0; a < 3; ++a) {
            float inv_dir = 1.0f / ray.dir[a];
            float t0 = (min[a] - ray.origin[a]) * inv_dir;
            float t1 = (max[a] - ray.origin[a]) * inv_dir;
            if (inv_dir < 0.0f) std::swap(t0, t1);
            tmin = fmax_(tmin, t0);
            tmax = fmin_(tmax, t1);
            if (!(tmax > tmin)) return false;
        }
        return true;
    }
    AABB expand(const AABB& o) const {  // aabb.rs:52-57
        return AABB{min_by_component(min, o.min), max_by_component(max, o.max)};
    }
    Vec3 center() const { return 0.5f * min + 0.5f * max; }  // aabb.rs:59-61
    AABB expand_to_point(Vec3 p) const {                    // aabb.rs:63-68
        return AABB{min_by_component(min, p), max_by_component(max, p)};
    }
};

// ------------------------------------------------------------------------------------------------
// render.rs:35-47  RaycastHit / Hitable.  obj_id / prim_id are instrumentation for the first-hit gate.
// ------------------------------------------------------------------------------------------------
struct RaycastHit {
    float t;
    Vec3 point, normal;
    int material;
    Vec2 uv;
    int obj_id = -1;   // render-object index (filled by RenderObjectInternal)
    int prim_id = 0;   // triangle index / Rect3d face index
};
struct Hitable {
    virtual ~Hitable() {}
    virtual bool hit(const Ray& r, float t_min, float t_max, Rng& rand, RaycastHit& out) const = 0;
    virtual AABB bounding_box() const = 0;
};

// ------------------------------------------------------------------------------------------------
// objects/mod.rs:19-31  solve_quadratic.  Returns count (0,1,2) with roots in r[].
// ------------------------------------------------------------------------------------------------
static inline int solve_quadratic(float a, float b, float c, float r[2]) {
    float disc = b * b - 4.0f * a * c;
    if (disc < 0.0f) {
        return 0;
    } else if (disc == 0.0f) {
        r[0] = -b / (2.0f * a);
        return 1;
    } else if (disc > 0.0f) {
        r[0] = (-b - std::sqrt(disc)) / (2.0f * a);
        r[1] = (-b + std::sqrt(disc)) / (2.0f * a);
        return 2;
    } else {
        // disc is NaN: Rust's `disc < 0.` and `disc == 0.` are both false -> falls to the else arm,
        // giving two NaN roots (which then fail every interval test).
        r[0] = (-b - std::sqrt(disc)) / (2.0f * a);
        r[1] = (-b + std::sqrt(disc)) / (2.0f * a);
        return 2;
    }
}

// sphere.rs:22-29
static inline Vec2 sphere_uv(Vec3 p) {
    float phi = std::atan2(p.z, p.x);
    float theta = std::asin(p.y);
    float u = 1.0f - (phi + PI_F) / (2.0f * PI_F);
    float v = (theta + PI_F / 2.0f) / PI_F;
    return Vec2{u, v};
}

// sphere.rs:32-65
struct Sphere : Hitable {
    float radius;
    int material;
    bool hit(const Ray& r, float t_min, float t_max, Rng&, RaycastHit& out) const override {
        ++g_cnt.prim_tests;
        ++g_cnt.sphere;
        Vec3 o = r.origin, d = r.dir;
        float a = dot(d, d);
        float b = 2.0f * dot(o, d);
        float c = dot(o, o) - radius * radius;
        float rt[2];
        int n = solve_quadratic(a, b, c, rt);
        if (n == 0) return false;
        float t;
        if (rt[0] < t_max && rt[0] > t_min) {
            t = rt[0];
        } else if (n == 2 && rt[1] < t_max && rt[1] > t_min) {
            t = rt[1];
        } else {
            return false;
        }
        Vec3 point = r.point(t);
        out.t = t;
        out.point = point;
        out.normal = point / radius;
        out.material = material;
        out.uv = sphere_uv(point / radius);
        out.prim_id = 0;
        return true;
    }
    AABB bounding_box() const override {  // sphere.rs:62-64
        return AABB{v3(-1.0f, -1.0f, -1.0f) * radius, v3(1.0f, 1.0f, 1.0f) * radius};
    }
};

// rect.rs:13-87  AARect<A1,A2>; `other` axis per util.rs:86-93.
struct AARect : Hitable {
    int a1, a2, ak;  // XY: (0,1,2)  XZ: (0,2,1)  YZ: (1,2,0)
    Vec2 min, max;
    float k;
    bool flip_normal;
    int material;
    bool hit(const Ray& r, float t_min, float t_max, Rng&, RaycastHit& out) const override {
        ++g_cnt.prim_tests;
        ++g_cnt.rect;
        float t = (k - r.origin[ak]) / r.dir[ak];
        if (t < t_min || t > t_max) return false;
        Vec3 point = r.point(t);
        if (point[a1] < min.x || point[a1] > max.x || point[a2] < min.y || point[a2] > max.y) return false;
        Vec3 normal = v3(ak == 0 ? 1.0f : 0.0f, ak == 1 ? 1.0f : 0.0f, ak == 2 ? 1.0f : 0.0f);
        out.t = t;
        out.point = point;
        out.normal = flip_normal ? -normal : normal;
        out.material = material;
        out.uv = Vec2{(point[a1] - min.x) / (max.x - min.x), (point[a2] - min.y) / (max.y - min.y)};
        out.prim_id = 0;
        return true;
    }
    AABB bounding_box() const override {  // rect.rs:75-86
        Vec3 lo = v3(0, 0, 0), hi = v3(0, 0, 0);
        lo.at(a1) = min.x; lo.at(a2) = min.y; lo.at(ak) = k - 0.01f;
        hi.at(a1) = max.x; hi.at(a2) = max.y; hi.at(ak) = k + 0.01f;
        return AABB{lo, hi};
    }
};

// rect3d.rs:10-105
struct Rect3d : Hitable {
    Vec3 pos, size;
    std::vector<AARect> faces;
    bool hit(const Ray& r, float t_min, float t_max, Rng& rand, RaycastHit& out) const override {
        bool any = false;
        float closest = t_max;
        for (size_t i = 0; i < faces.size(); ++i) {
            RaycastHit h;
            if (faces[i].hit(r, t_min, closest, rand, h)) {
                closest = h.t;
                out = h;
                out.prim_id = (int)i;
                any = true;
            }
        }
        return any;
    }
    AABB bounding_box() const override { return AABB{pos, pos + size}; }  // rect3d.rs:102-104
};

// disk.rs:40-91
struct Disk : Hitable {
    float radius, phi_max, inner_radius;
    int material;
    bool hit(const Ray& r, float t_min, float t_max, Rng&, RaycastHit& out) const override {
        ++g_cnt.prim_tests;
        ++g_cnt.conic;
        if (r.dir.y == 0.0f) return false;
        float t = -r.origin.y / r.dir.y;
        if (t < t_min || t > t_max) return false;
        Vec3 point = r.point(t);
        float dist2 = point.x * point.x + point.z * point.z;
        if (dist2 > radius * radius || dist2 < inner_radius * inner_radius) return false;
        float phi = std::atan2(point.z, point.x);
        if (phi < 0.0f) phi = phi + 2.0f * PI_F;
        if (phi > phi_max) return false;
        float u = phi / phi_max;
        float dist = std::sqrt(dist2);
        float v = 1.0f - (dist - inner_radius) / (radius - inner_radius);
        out.t = t;
        out.point = point;
        out.normal = v3(0, 1, 0);
        out.material = material;
        out.uv = Vec2{u, v};
        out.prim_id = 0;
        return true;
    }
    AABB bounding_box() const override {  // disk.rs:85-90 (degenerate in x and z — preserved)
        return AABB{v3(-radius, 0.0f, radius), v3(-radius, 0.001f, radius)};
    }
};

// cylinder.rs:41-98
struct Cylinder : Hitable {
    float radius, height, max_phi;
    int material;
    bool check_solution(const Ray& r, float t, float t_min, float t_max, RaycastHit& out) const {
        if (t > t_max || t < t_min) return false;
        Vec3 point = r.point(t);
        float phi = std::atan2(point.z, point.x);
        if (phi < 0.0f) phi = phi + PI_F * 2.0f;
        if (point.y > 0.0f && point.y < height && phi < max_phi) {
            out.t = t;
            out.point = point;
            out.normal = v3(point.x / radius, 0.0f, point.z / radius);
            out.material = material;
            out.uv = Vec2{phi / max_phi, point.y / height};
            out.prim_id = 0;
            return true;
        }
        return false;
    }
    bool hit(const Ray& r, float t_min, float t_max, Rng&, RaycastHit& out) const override {
        ++g_cnt.prim_tests;
        ++g_cnt.conic;
        Vec3 o = r.origin, d = r.dir;
        float a = d.x * d.x + d.z * d.z;
        float b = 2.0f * (d.x * o.x + d.z * o.z);
        float c = o.x * o.x + o.z * o.z - radius * radius;
        float disc = b * b - 4.0f * a * c;
        if (disc > 0.0f) {
            float rt[2];
            int n = solve_quadratic(a, b, c, rt);
            if (n >= 1) {
                if (check_solution(r, rt[0], t_min, t_max, out)) return true;
                if (n == 2) return check_solution(r, rt[1], t_min, t_max, out);
            }
        }
        return false;
    }
    AABB bounding_box() const override {  // cylinder.rs:92-97
        return AABB{v3(-radius, 0.0f, -radius), v3(radius, height, radius)};
    }
};

// cone.rs:27-96
struct Cone : Hitable {
    float radius, height;
    int material;
    bool check_solution(const Ray& r, float t, float t_min, float t_max, RaycastHit& out) const {
        if (t > t_max || t < t_min) return false;
        Vec3 point = r.point(t);
        if (point.y < 0.0f || point.y > height) return false;
        float v = point.y / height;
        float phi = std::acos(point.x / (radius * (1.0f - v)));
        float u = phi / (2.0f * PI_F);
        Vec3 dpdu = v3(-point.z, 0.0f, point.x);
        Vec3 dpdv = v3(-point.x / (1.0f - v), height, -point.z / (1.0f - v));
        out.t = t;
        out.point = point;
        out.normal = normalized(cross(dpdv, dpdu));
        out.material = material;
        out.uv = Vec2{u, v};
        out.prim_id = 0;
        return true;
    }
    bool hit(const Ray& r, float t_min, float t_max, Rng&, RaycastHit& out) const override {
        ++g_cnt.prim_tests;
        ++g_cnt.conic;
        Vec3 o = r.origin, d = r.dir;
        float r2_div_h2 = radius * radius / (height * height);
        float a = d.x * d.x + d.z * d.z - r2_div_h2 * d.y * d.y;
        float b = 2.0f * (d.x * o.x + d.z * o.z - r2_div_h2 * d.y * (o.y - height));
        float c = o.x * o.x + o.z * o.z - r2_div_h2 * (o.y - height) * (o.y - height);
        float rt[2];
        int n = solve_quadratic(a, b, c, rt);
        if (n >= 1) {
            if (check_solution(r, rt[0], t_min, t_max, out)) return true;
            if (n == 2) return check_solution(r, rt[1], t_min, t_max, out);
        }
        return false;
    }
    AABB bounding_box() const override {  // cone.rs:90-95
        return AABB{v3(-radius, 0.0f, -radius), v3(radius, height, radius)};
    }
};

// util.rs:104-118  (signed comparison, not |d|)
static inline int max_component_idx(Vec3 v) {
    if (v.x > v.y) {
        return (v.z > v.x) ? 2 : 0;
    } else {
        return (v.z > v.y) ? 2 : 1;
    }
}

// mesh.rs:12-110
struct TriangleMesh {
    std::vector<uint32_t> indicies;
    std::vector<Vec3> verts;
    bool has_normals = false, has_uvs = false;
    std::vector<Vec3> normals;
    std::vector<Vec2> uvs;
    int material = 0;
    size_t num_tris() const { return indicies.size() / 3; }
};

// mesh.rs:112-242
struct Triangle {
    const TriangleMesh* mesh;
    size_t index;
    bool hit(const Ray& r, float t_min, float t_max, Rng&, RaycastHit& out) const {
        ++g_cnt.prim_tests;
        ++g_cnt.tri;
        const TriangleMesh& m = *mesh;
        size_t base = 3 * index;
        Vec3 p0 = m.verts[m.indicies[base]], p1 = m.verts[m.indicies[base + 1]],
             p2 = m.verts[m.indicies[base + 2]];
        Vec3 p0t = p0 - r.origin, p1t = p1 - r.origin, p2t = p2 - r.origin;
        Vec3 d = r.dir;
        int kz = max_component_idx(d);
        int kx = (kz + 1) % 3;
        int ky = (kx + 1) % 3;
        d = v3(d[kx], d[ky], d[kz]);
        p0t = v3(p0t[kx], p0t[ky], p0t[kz]);
        p1t = v3(p1t[kx], p1t[ky], p1t[kz]);
        p2t = v3(p2t[kx], p2t[ky], p2t[kz]);
        float sx = -d.x / d.z;
        float sy = -d.y / d.z;
        float sz = 1.0f / d.z;
        p0t.x += sx * p0t.z; p0t.y += sy * p0t.z;
        p1t.x += sx * p1t.z; p1t.y += sy * p1t.z;
        p2t.x += sx * p2t.z; p2t.y += sy * p2t.z;
        float e0 = p1t.x * p2t.y - p1t.y * p2t.x;
        float e1 = p2t.x * p0t.y - p2t.y * p0t.x;
        float e2 = p0t.x * p1t.y - p0t.y * p1t.x;
        if ((e0 < 0.0f || e1 < 0.0f || e2 < 0.0f) && (e0 > 0.0f || e1 > 0.0f || e2 > 0.0f)) return false;
        float det = e0 + e1 + e2;
        if (det == 0.0f) return false;
        p0t.z *= sz; p1t.z *= sz; p2t.z *= sz;
        float t_scaled = e0 * p0t.z + e1 * p1t.z + e2 * p2t.z;
        if (det < 0.0f && (t_scaled >= t_min * det || t_scaled < t_max * det)) {
            return false;
        } else if (det > 0.0f && (t_scaled <= t_min * det || t_scaled > t_max * det)) {
            return false;
        }
        float inv_det = 1.0f / det;
        float b0 = e0 * inv_det, b1 = e1 * inv_det, b2 = e2 * inv_det;
        float t = t_scaled * inv_det;
        Vec3 point = b0 * p0 + b1 * p1 + b2 * p2;
        Vec2 uv0{0, 0}, uv1{1, 0}, uv2{0, 1};  // mesh.rs:108 default uvs
        if (m.has_uvs) {
            uv0 = m.uvs[m.indicies[base]]; uv1 = m.uvs[m.indicies[base + 1]]; uv2 = m.uvs[m.indicies[base + 2]];
        }
        Vec2 uv = b0 * uv0 + b1 * uv1 + b2 * uv2;
        Vec3 normal;
        if (m.has_normals) {
            Vec3 n0 = m.normals[m.indicies[base]], n1 = m.normals[m.indicies[base + 1]],
                 n2 = m.normals[m.indicies[base + 2]];
            normal = normalized(b0 * n0 + b1 * n1 + b2 * n2);
        } else {
            normal = cross(p0 - p2, p1 - p2);  // NOT normalised (mesh.rs:209)
        }
        out.t = t;
        out.point = point;
        out.normal = normal;
        out.material = m.material;
        out.uv = uv;
        out.prim_id = (int)index;
        return true;
    }
    AABB bounding_box() const {  // mesh.rs:221-242
        const TriangleMesh& m = *mesh;
        size_t base = 3 * index;
        Vec3 p0 = m.verts[m.indicies[base]], p1 = m.verts[m.indicies[base + 1]],
             p2 = m.verts[m.indicies[base + 2]];
        AABB aabb = AABB::from_two_points(p0, p1).expand_to_point(p2);
        Vec3 size = aabb.max - aabb.min;
        size = v3(std::fabs(size.x), std::fabs(size.y), std::fabs(size.z));
        if (size.x < 0.001f) { aabb.min.x -= 0.001f; aabb.max.x += 0.001f; }
        if (size.y < 0.001f) { aabb.min.y -= 0.001f; aabb.max.y += 0.001f; }
        if (size.z < 0.001f) { aabb.min.z -= 0.001f; aabb.max.z += 0.001f; }
        return aabb;
    }
};

// ------------------------------------------------------------------------------------------------
// bvh.rs — generic over the item type via two small adaptor functions.
// ------------------------------------------------------------------------------------------------
struct RenderObjectInternal;
static bool item_hit(const RenderObjectInternal* const& it, const Ray& r, float t_min, float t_max, Rng& rand,
                     RaycastHit& out);
static AABB item_bbox(const RenderObjectInternal* const& it);
static inline bool item_hit(const Triangle& it, const Ray& r, float t_min, float t_max, Rng& rand, RaycastHit& out) {
    return it.hit(r, t_min, t_max, rand, out);
}
static inline AABB item_bbox(const Triangle& it) { return it.bounding_box(); }

template <class T>
struct BVHNode {
    enum Kind { LEAF, DOUBLE_LEAF, BRANCH } kind;
    T a, b;                              // items for LEAF / DOUBLE_LEAF
    std::unique_ptr<BVHNode<T>> l, r;    // children for BRANCH
    AABB aabb;

    // bvh.rs:115-151 — both children are ALWAYS visited with the same t_max; ties go to the right.
    bool hit(const Ray& ray, float t_min, float t_max, Rng& rand, RaycastHit& out) const {
        if (!aabb.hit(ray, t_min, t_max)) return false;
        switch (kind) {
            case LEAF:
                return item_hit(a, ray, t_min, t_max, rand, out);
            case DOUBLE_LEAF: {
                RaycastHit lh, rh;
                bool lhit = item_hit(a, ray, t_min, t_max, rand, lh);
                bool rhit = item_hit(b, ray, t_min, t_max, rand, rh);
                if (!lhit && !rhit) return false;
                if (lhit && !rhit) { out = lh; return true; }
                if (!lhit && rhit) { out = rh; return true; }
                if (lh.t < rh.t) out = lh; else out = rh;
                return true;
            }
            default: {
                RaycastHit lh, rh;
                bool lhit = l->hit(ray, t_min, t_max, rand, lh);
                bool rhit = r->hit(ray, t_min, t_max, rand, rh);
                if (!lhit && !rhit) return false;
                if (lhit && !rhit) { out = lh; return true; }
                if (!lhit && rhit) { out = rh; return true; }
                if (lh.t < rh.t) out = lh; else out = rh;
                return true;
            }
        }
    }
};

// bvh.rs:21-71  new_helper.  `items(i)` yields the aggregate's i-th item.
template <class T, class GetItem>
static std::unique_ptr<BVHNode<T>> bvh_new_helper(const GetItem& items, size_t* indicies, size_t n, size_t depth) {
    int axis = (int)(depth % 3);
    // indicies.sort_by(...) — Rust's slice::sort_by is a stable sort; boxes recomputed per comparison.
    std::stable_sort(indicies, indicies + n, [&](size_t x, size_t y) {
        float cx = item_bbox(items(x)).center()[axis];
        float cy = item_bbox(items(y)).center()[axis];
        return cx < cy;
    });
    auto node = std::make_unique<BVHNode<T>>();
    if (n == 1) {
        node->kind = BVHNode<T>::LEAF;
        node->a = items(indicies[0]);
        node->b = node->a;
        node->aabb = item_bbox(node->a);
    } else if (n == 2) {
        node->kind = BVHNode<T>::DOUBLE_LEAF;
        node->a = items(indicies[0]);
        node->b = items(indicies[1]);
        node->aabb = item_bbox(node->a).expand(item_bbox(node->b));
    } else {
        size_t half = n / 2;
        node->kind = BVHNode<T>::BRANCH;
        node->l = bvh_new_helper<T>(items, indicies, half, depth + 1);
        node->r = bvh_new_helper<T>(items, indicies + half, n - half, depth + 1);
        node->aabb = node->l->aabb.expand(node->r->aabb);
    }
    return node;
}

// mesh.rs:21-30: TriangleMesh::to_hitable() == BVHNode<Triangle> built over the mesh's triangles.
struct MeshBVH : Hitable {
    std::shared_ptr<TriangleMesh> mesh;
    std::unique_ptr<BVHNode<Triangle>> root;
    void build() {
        size_t n = mesh->num_tris();
        std::vector<size_t> idx(n);
        for (size_t i = 0; i < n; ++i) idx[i] = i;
        const TriangleMesh* mp = mesh.get();
        auto get = [mp](size_t i) { return Triangle{mp, i}; };
        root = bvh_new_helper<Triangle>(get, idx.data(), n, 0);
    }
    bool hit(const Ray& r, float t_min, float t_max, Rng& rand, RaycastHit& out) const override {
        return root->hit(r, t_min, t_max, rand, out);
    }
    AABB bounding_box() const override { return root->aabb; }
};

// volume.rs:57-87
struct ConstantMedium : Hitable {
    std::unique_ptr<Hitable> obj;
    float density;
    int material;
    int rng_id = 0;  // render-object index: keys the free-path draw (see Rng::rand_keyed)
    bool hit(const Ray& r, float t_min, float t_max, Rng& rand, RaycastHit& out) const override {
        const float FMAX = 3.40282347e+38f;
        RaycastHit rec1, rec2;
        if (obj->hit(r, -FMAX, FMAX, rand, rec1)) {
            if (obj->hit(r, rec1.t + 0.0001f, FMAX, rand, rec2)) {
                rec1.t = fmax_(rec1.t, t_min);
                rec2.t = fmin_(rec2.t, t_max);
                if (rec1.t >= rec2.t) return false;
                rec1.t = fmax_(rec1.t, 0.0f);
                float dist_inside_boundary = (rec2.t - rec1.t) * mag(r.dir);
                float hit_distance = -(1.0f / density) * std::log10(rand.rand_keyed((uint32_t)rng_id));
                if (hit_distance < dist_inside_boundary) {
                    float t = rec1.t + hit_distance / mag(r.dir);
                    out.t = t;
                    out.point = r.point(t);
                    out.normal = v3(0, 1, 0);
                    out.material = material;
                    out.uv = Vec2{0, 0};
                    out.prim_id = 0;
                    return true;
                }
            }
        }
        return false;
    }
    AABB bounding_box() const override { return obj->bounding_box(); }
};

// ------------------------------------------------------------------------------------------------
// scene.rs:151-292  RenderObjectInternal
// ------------------------------------------------------------------------------------------------
struct RenderObjectInternal {
    std::unique_ptr<Hitable> obj;
    Vec3 position;
    Mat3 rotation_mat, inv_rotation_mat;
    bool flip_normals;
    AABB aabb;
    int id;

    float cos_trace() const {  // scene.rs:181-185 / 242-245
        float trace = rotation_mat.cols[0].x + rotation_mat.cols[1].y + rotation_mat.cols[2].z;
        return 0.5f * (trace - 1.0f);
    }
    void update_bounding_box() {  // scene.rs:167-212
        AABB bbox = obj->bounding_box();
        AABB rotated;
        if (cos_trace() < 0.999f) {
            Vec3 mn = 10e9f * v3(1, 1, 1);
            Vec3 mx = -10e9f * v3(1, 1, 1);
            for (int i = 0; i < 2; ++i)
                for (int j = 0; j < 2; ++j)
                    for (int k = 0; k < 2; ++k) {
                        float x = i == 0 ? bbox.min.x : bbox.max.x;
                        float y = j == 0 ? bbox.min.y : bbox.max.y;
                        float z = k == 0 ? bbox.min.z : bbox.max.z;
                        Vec3 np = rotation_mat * v3(x, y, z);
                        for (int c = 0; c < 3; ++c) {
                            mx.at(c) = fmax_(np[c], mx[c]);
                            mn.at(c) = fmin_(np[c], mn[c]);
                        }
                    }
            rotated = AABB{mn, mx};
        } else {
            rotated = bbox;
        }
        aabb = AABB{rotated.min + position, rotated.max + position};
    }
    // scene.rs:235-266  render_object_internet_hit
    bool hit(const Ray& r, float t_min, float t_max, Rng& rand, RaycastHit& out) const {
        Ray new_ray;
        if (cos_trace() < 0.999f) {
            ++g_cnt.xform_rot;
            new_ray = Ray{inv_rotation_mat * (r.origin - position), inv_rotation_mat * r.dir};
        } else {
            ++g_cnt.xform_trans;
            new_ray = Ray{r.origin - position, r.dir};
        }
        if (obj->hit(new_ray, t_min, t_max, rand, out)) {
            out.point = rotation_mat * out.point;
            out.point = out.point + position;
            out.normal = rotation_mat * out.normal;
            if (flip_normals) out.normal = -out.normal;
            out.obj_id = id;
            return true;
        }
        return false;
    }
};
static bool item_hit(const RenderObjectInternal* const& it, const Ray& r, float t_min, float t_max, Rng& rand,
                     RaycastHit& out) {
    return it->hit(r, t_min, t_max, rand, out);
}
static AABB item_bbox(const RenderObjectInternal* const& it) { return it->aabb; }

// ------------------------------------------------------------------------------------------------
// texture.rs
// ------------------------------------------------------------------------------------------------
struct Texture {
    virtual ~Texture() {}
    virtual Vec3 sample(Vec2 uv, const Vec3& point) const = 0;
};
struct ConstantTexture : Texture {  // texture.rs:29-34
    Vec3 color;
    Vec3 sample(Vec2, const Vec3&) const override { return color; }
};
struct CheckerTexture : Texture {  // texture.rs:57-73
    const Texture *odd, *even;
    float scale;
    Vec3 sample(Vec2 uv, const Vec3& point) const override {
        // iter().map(|x| (scale*x).sin()).product::<f32>() : fold starting at 1.0
        float sx = std::sin(scale * point.x), sy = std::sin(scale * point.y), sz = std::sin(scale * point.z);
        float prod = 1.0f;
        prod = prod * sx;
        prod = prod * sy;
        prod = prod * sz;
        // A product of two NaNs is one of them, chosen by the operand order of the multiply instruction, which the
        // compiler picks (this file's -O2 and -O3 builds differ).  Pin it: the first NaN factor in x, y, z order decides.
        if (std::isnan(prod)) prod = std::isnan(sx) ? sx : (std::isnan(sy) ? sy : sz);
        if (!std::signbit(prod)) return even->sample(uv, point);
        return odd->sample(uv, point);
    }
};
// texture.rs:80-106 — Ken Perlin's reference permutation (a published constant), doubled at load.
static const uint8_t PERLIN_P256[256] = {
    151, 160, 137, 91,  90,  15,  131, 13,  201, 95,  96,  53,  194, 233, 7,   225, 140, 36,  103, 30,  69,  142,
    8,   99,  37,  240, 21,  10,  23,  190, 6,   148, 247, 120, 234, 75,  0,   26,  197, 62,  94,  252, 219, 203,
    117, 35,  11,  32,  57,  177, 33,  88,  237, 149, 56,  87,  174, 20,  125, 136, 171, 168, 68,  175, 74,  165,
    71,  134, 139, 48,  27,  166, 77,  146, 158, 231, 83,  111, 229, 122, 60,  211, 133, 230, 220, 105, 92,  41,
    55,  46,  245, 40,  244, 102, 143, 54,  65,  25,  63,  161, 1,   216, 80,  73,  209, 76,  132, 187, 208, 89,
    18,  169, 200, 196, 135, 130, 116, 188, 159, 86,  164, 100, 109, 198, 173, 186, 3,   64,  52,  217, 226, 250,
    124, 123, 5,   202, 38,  147, 118, 126, 255, 82,  85,  212, 207, 206, 59,  227, 47,  16,  58,  17,  182, 189,
    28,  42,  223, 183, 170, 213, 119, 248, 152, 2,   44,  154, 163, 70,  221, 153, 101, 155, 167, 43,  172, 9,
    129, 22,  39,  253, 19,  98,  108, 110, 79,  113, 224, 232, 178, 185, 112, 104, 218, 246, 97,  228, 251, 34,
    242, 193, 238, 210, 144, 12,  191, 179, 162, 241, 81,  51,  145, 235, 249, 14,  239, 107, 49,  192, 214, 31,
    181, 199, 106, 157, 184, 84,  204, 176, 115, 121, 50,  45,  127, 4,   150, 254, 138, 236, 205, 93,  222, 114,
    67,  29,  24,  72,  243, 141, 128, 195, 78,  66,  215, 61,  156, 180};
static inline uint64_t PERLIN_P(uint64_t i) { return PERLIN_P256[i & 255]; }  // P[512] = P256 ++ P256

static inline float perlin_fade(float t) { return t * t * (3.0f - 2.0f * t); }  // texture.rs:163-166
static inline float perlin_grad(uint64_t hash, float x, float y, float z) {    // texture.rs:168-182
    uint64_t h = hash & 15;
    float u = h < 8 ? x : y;
    float v = h < 4 ? y : ((h == 12 || h == 14) ? x : z);
    u = (h & 1) == 0 ? u : -u;
    v = (h & 2) == 0 ? v : -v;
    return u + v;
}
static inline float perlin_lerp(float t, float a, float b) { return a + t * (b - a); }  // texture.rs:184-186
static float perlin_noise(Vec3 p) {  // texture.rs:113-158
    uint64_t x0 = f32_as_usize(std::floor(p.x)) & 255;
    uint64_t y0 = f32_as_usize(std::floor(p.y)) & 255;
    uint64_t z0 = f32_as_usize(std::floor(p.z)) & 255;
    float x = p.x - std::floor(p.x);
    float y = p.y - std::floor(p.y);
    float z = p.z - std::floor(p.z);
    float u = perlin_fade(x), v = perlin_fade(y), w = perlin_fade(z);
    uint64_t a = PERLIN_P(x0) + y0;
    uint64_t aa = PERLIN_P(a) + z0;
    uint64_t ab = PERLIN_P(a + 1) + z0;
    uint64_t b = PERLIN_P(x0 + 1) + y0;
    uint64_t ba = PERLIN_P(b) + z0;
    uint64_t bb = PERLIN_P(b + 1) + z0;
    return perlin_lerp(
        w,
        perlin_lerp(v,
                    perlin_lerp(u, perlin_grad(PERLIN_P(aa), x, y, z), perlin_grad(PERLIN_P(ba), x - 1.0f, y, z)),
                    perlin_lerp(u, perlin_grad(PERLIN_P(ab), x, y - 1.0f, z),
                                perlin_grad(PERLIN_P(bb), x - 1.0f, y - 1.0f, z))),
        perlin_lerp(v,
                    perlin_lerp(u, perlin_grad(PERLIN_P(aa + 1), x, y, z - 1.0f),
                                perlin_grad(PERLIN_P(ba + 1), x - 1.0f, y, z - 1.0f)),
                    perlin_lerp(u, perlin_grad(PERLIN_P(ab + 1), x, y - 1.0f, z - 1.0f),
                                perlin_grad(PERLIN_P(bb + 1), x - 1.0f, y - 1.0f, z - 1.0f))));
}
struct PerlinNoiseTexture : Texture {  // texture.rs:160-167 (sample)
    float scale;
    Vec3 sample(Vec2, const Vec3& point) const override {
        float a = perlin_noise(point * scale);
        return v3(1, 1, 1) * fmin_(a + 0.5f, 1.0f);
    }
};
static float turb(uint64_t depth, Vec3 point) {  // texture.rs:206-217 (no abs)
    float accum = 0.0f;
    Vec3 p = point;
    float weight = 1.0f;
    for (uint64_t i = 0; i < depth; ++i) {
        float a = perlin_noise(p);
        accum += weight * a;
        weight *= 0.5f;
        p = p * 2.0f;
    }
    return accum;
}
struct TurbulenceTexture : Texture {  // texture.rs:219-224
    uint64_t depth;
    float scale;
    Vec3 sample(Vec2, const Vec3& point) const override { return v3(1, 1, 1) * turb(depth, point * scale); }
};
struct MarbleTexture : Texture {  // texture.rs:239-249
    uint64_t depth;
    float scale;
    Vec3 sample(Vec2, const Vec3& point) const override {
        // Vec3::one() * 0.5 * (1. + sin(scale*z + 10.*turb))  — left-assoc: (one*0.5) * (...)
        Vec3 half = v3(1, 1, 1) * 0.5f;
        return half * (1.0f + std::sin(scale * point.z + 10.0f * turb(depth, point)));
    }
};
struct ImageTexture : Texture {  // texture.rs:294-310 — texels decoded once by the harness (RGBA8)
    uint32_t w, h;
    std::vector<uint8_t> rgba;
    Vec3 sample(Vec2 uv, const Vec3&) const override {
        float fi = uv.x * (float)w;
        float fj = (1.0f - uv.y) * (float)h;
        uint32_t i = std::min(std::max(f32_as_u32(fi), 0u), w - 1);
        uint32_t j = std::min(std::max(f32_as_u32(fj), 0u), h - 1);
        const uint8_t* c = &rgba[4 * ((size_t)j * w + i)];
        return v3((float)c[0], (float)c[1], (float)c[2]) / 255.0f;
    }
};

// ------------------------------------------------------------------------------------------------
// util.rs:36-73
// ------------------------------------------------------------------------------------------------
static Vec3 random_in_unit_sphere(Rng& rng) {
    for (;;) {
        float a = rng.rand_f32(), b = rng.rand_f32(), c = rng.rand_f32();
        Vec3 p = 2.0f * v3(a, b, c) - v3(1, 1, 1);
        if (mag_sq(p) < 1.0f) return p;
    }
}
static Vec3 random_in_unit_disk(Rng& rng) {
    for (;;) {
        float a = rng.rand_f32(), b = rng.rand_f32();
        Vec3 p = 2.0f * v3(a, b, 0.0f) - v3(1.0f, 1.0f, 0.0f);
        if (dot(p, p) < 1.0f) return p;
    }
}
static inline Vec3 reflect(Vec3 v, Vec3 n) { return v - 2.0f * dot(v, n) * n; }  // (2*v.n)*n
static inline bool refract(Vec3 v, Vec3 n, float ni_over_nt, Vec3& out) {
    Vec3 uv = normalized(v);
    float dt = dot(uv, n);
    float disc = 1.0f - ni_over_nt * ni_over_nt * (1.0f - dt * dt);
    if (disc > 0.0f) {
        out = ni_over_nt * (uv - n * dt) - n * std::sqrt(disc);
        return true;
    }
    return false;
}
static inline float schlick(float cosine, float ref_idx) {
    float r0 = (1.0f - ref_idx) / (1.0f + ref_idx);
    r0 = r0 * r0;
    return r0 + (1.0f - r0) * std::pow(1.0f - cosine, 5.0f);
}

// ------------------------------------------------------------------------------------------------
// material.rs
// ------------------------------------------------------------------------------------------------
struct ScatterResult {
    Vec3 attenuation;
    Ray scattered;
};
struct Material {
    virtual ~Material() {}
    virtual bool scatter(const Ray& r_in, const RaycastHit& hit, Rng& rand, ScatterResult& out) const = 0;
    virtual Vec3 emit(Vec2, const Vec3&) const { return v3(0, 0, 0); }  // material.rs:13-15
};
struct LambertianMat : Material {  // material.rs:63-75
    const Texture* albedo;
    bool scatter(const Ray&, const RaycastHit& hit, Rng& rand, ScatterResult& out) const override {
        Vec3 target = hit.point + hit.normal + random_in_unit_sphere(rand);
        out.scattered = Ray{hit.point, target - hit.point};
        out.attenuation = albedo->sample(hit.uv, hit.point);
        return true;
    }
};
struct MetalMat : Material {  // material.rs:89-107
    Vec3 albedo;
    float roughness;
    bool scatter(const Ray& r_in, const RaycastHit& hit, Rng& rand, ScatterResult& out) const override {
        Vec3 reflected = reflect(r_in.dir, hit.normal);
        out.scattered = Ray{hit.point, reflected + roughness * random_in_unit_sphere(rand)};
        out.attenuation = albedo;
        return dot(out.scattered.dir, hit.normal) > 0.0f;
    }
};
struct DielectricMat : Material {  // material.rs:120-151
    float ref_idx;
    bool scatter(const Ray& r_in, const RaycastHit& hit, Rng& rand, ScatterResult& out) const override {
        Vec3 reflected = reflect(r_in.dir, hit.normal);
        Vec3 outward_normal;
        float ni_over_nt, cosine;
        if (dot(r_in.dir, hit.normal) > 0.0f) {
            outward_normal = -hit.normal;
            ni_over_nt = ref_idx;
            cosine = ref_idx * dot(r_in.dir, hit.normal) / mag(r_in.dir);
        } else {
            outward_normal = hit.normal;
            ni_over_nt = 1.0f / ref_idx;
            cosine = -dot(r_in.dir, hit.normal) / mag(r_in.dir);
        }
        Vec3 refracted;
        if (refract(r_in.dir, outward_normal, ni_over_nt, refracted)) {
            if (rand.rand_f32() > schlick(cosine, ref_idx)) {
                out.scattered = Ray{hit.point, refracted};
                out.attenuation = v3(1, 1, 1);
                return true;
            }
        }
        out.scattered = Ray{hit.point, reflected};
        out.attenuation = v3(1, 1, 1);
        return true;
    }
};
struct EmissiveMat : Material {  // material.rs:172-181
    const Texture* albedo;
    bool scatter(const Ray&, const RaycastHit&, Rng&, ScatterResult&) const override { return false; }
    Vec3 emit(Vec2 uv, const Vec3& point) const override { return albedo->sample(uv, point); }
};
struct IsotropicMat : Material {  // material.rs:196-204
    const Texture* texture;
    bool scatter(const Ray&, const RaycastHit& hit, Rng& rand, ScatterResult& out) const override {
        out.attenuation = texture->sample(hit.uv, hit.point);
        out.scattered = Ray{hit.point, random_in_unit_sphere(rand)};
        return true;
    }
};

// ------------------------------------------------------------------------------------------------
// environment.rs (+ examples/hdri_test.rs:14-20, 72-81)
// ------------------------------------------------------------------------------------------------
struct Environment {
    virtual ~Environment() {}
    virtual Vec3 sample(Vec3 dir) const = 0;
};
struct ColorEnv : Environment {  // environment.rs:21-26
    Vec3 color;
    Vec3 sample(Vec3) const override { return color; }
};
struct SkyEnv : Environment {  // environment.rs:60-67
    Vec3 zenith_color, horizon_color;
    Vec3 sample(Vec3 dir) const override {
        float t = 0.5f * (dir.y + 1.0f);
        return (1.0f - t) * horizon_color + t * zenith_color;
    }
};
struct HdrEnvironment : Environment {  // examples/hdri_test.rs:22-82
    std::vector<float> pixels;      // RGB f32, row-major
    float width, height;
    Vec3 sample(Vec3 dir) const override {
        Vec2 uv = sphere_uv(dir);
        uint64_t x = f32_as_usize(uv.x * width);
        uint64_t y = f32_as_usize((1.0f - uv.y) * height);
        uint64_t idx = f32_as_usize((float)y * width) + x;
        // DEVIATION (documented): the reference indexes out of bounds (panics) when dir.y == -1 or the
        // NaN/edge cases push idx past the end; both oracle and CUDA clamp to the last texel instead.
        uint64_t n = pixels.size() / 3;
        if (idx >= n) idx = n - 1;
        return v3(pixels[3 * idx], pixels[3 * idx + 1], pixels[3 * idx + 2]);
    }
};

// ------------------------------------------------------------------------------------------------
// camera.rs:74-116
// ------------------------------------------------------------------------------------------------
struct Camera {
    Vec3 position, horizontal, vertical, lower_left, u, v, w;
    float lens_radius;
    static Camera make(Vec3 cam_pos, Vec3 look_at, float vfov, float aperture, float focus_dist, size_t width,
                       size_t height) {
        float theta = vfov * PI_F / 180.0f;
        Vec3 w = normalized(cam_pos - look_at);
        Vec3 u = normalized(cross(v3(0, 1, 0), w));
        Vec3 v = cross(w, u);
        float half_height = std::tan(theta / 2.0f);
        float half_width = half_height * (float)width / (float)height;
        Camera c;
        c.lower_left = cam_pos - half_width * focus_dist * u - half_height * focus_dist * v - w * focus_dist;
        c.horizontal = 2.0f * half_width * focus_dist * u;
        c.vertical = 2.0f * half_height * focus_dist * v;
        c.position = cam_pos;
        c.u = u; c.v = v; c.w = w;
        c.lens_radius = aperture / 2.0f;
        return c;
    }
    Ray ray(float s, float t, Rng& rand) const {
        Vec3 rd = lens_radius * random_in_unit_disk(rand);
        Vec3 offset = u * rd.x + v * rd.y;
        return Ray{position + offset, lower_left + s * horizontal + t * vertical - position - offset};
    }
};

// ------------------------------------------------------------------------------------------------
// scene.rs:93-165  SceneInternal, plus the builder state for the C API.
// ------------------------------------------------------------------------------------------------
struct Scene : Hitable {
    std::vector<std::unique_ptr<Texture>> textures;
    std::vector<std::unique_ptr<Material>> materials;
    std::vector<int> material_kind;
    std::vector<std::unique_ptr<Hitable>> shapes;       // staging: moved into objects / media
    std::vector<std::shared_ptr<TriangleMesh>> meshes;  // keep-alive
    std::vector<std::unique_ptr<RenderObjectInternal>> render_objects;
    std::unique_ptr<Environment> environment;
    std::unique_ptr<BVHNode<const RenderObjectInternal*>> bvh;
    std::string error;

    // scene.rs:137-149 — linear scan with shrinking `closest`.
    bool hit(const Ray& r, float t_min, float t_max, Rng& rand, RaycastHit& out) const override {
        bool any = false;
        float closest = t_max;
        for (const auto& ro : render_objects) {
            RaycastHit h;
            if (ro->hit(r, t_min, closest, rand, h)) {
                closest = h.t;
                out = h;
                any = true;
            }
        }
        return any;
    }
    AABB bounding_box() const override {  // scene.rs:151-163
        AABB res = render_objects.at(0)->aabb;
        for (size_t i = 1; i < render_objects.size(); ++i) res = res.expand(render_objects[i]->aabb);
        return res;
    }
    void build_bvh() {  // bvh.rs:79-98
        size_t n = render_objects.size();
        std::vector<size_t> idx(n);
        for (size_t i = 0; i < n; ++i) idx[i] = i;
        auto get = [this](size_t i) -> const RenderObjectInternal* { return render_objects[i].get(); };
        bvh = bvh_new_helper<const RenderObjectInternal*>(get, idx.data(), n, 0);
    }
    bool root_hit(bool use_bvh, const Ray& r, float t_min, float t_max, Rng& rand, RaycastHit& out) const {
        if (use_bvh) return bvh->hit(r, t_min, t_max, rand, out);
        return hit(r, t_min, t_max, rand, out);
    }
};

// render.rs:12-33
static Vec3 color(const Ray& r, const Scene& scene, bool use_bvh, size_t depth, Rng& rand) {
    ++g_cnt.rays;
    RaycastHit hit;
    rand.set_stream((uint32_t)depth, STREAM_MEDIUM);
    if (scene.root_hit(use_bvh, r, 0.001f, 2e9f, rand, hit)) {
        const Material& m = *scene.materials[hit.material];
        Vec3 emit = m.emit(hit.uv, hit.point);
        if (depth < 10) {
            ScatterResult res;
            rand.set_stream((uint32_t)depth, STREAM_SCATTER);
            if (m.scatter(r, hit, rand, res)) {
                return emit + res.attenuation * color(res.scattered, scene, use_bvh, depth + 1, rand);
            } else {
                return emit;
            }
        } else {
            return emit;
        }
    } else {
        return scene.environment->sample(normalized(r.dir));
    }
}

struct RenderParams {  // mirrors Renderer + CameraSettings (render.rs:57-77, camera.rs:18-24)
    uint32_t width, height;
    uint32_t samples;       // total spp the image is normalised by
    uint32_t sample_begin;  // first sample index rendered by this call
    uint32_t sample_count;  // number of samples rendered by this call
    uint32_t use_bvh;
    float gamma;
    float cam_pos[3], look_at[3];
    float vfov, aperture, focus_dist;
    uint64_t seed;
};

static Camera make_camera(const RenderParams& p) {
    return Camera::make(v3(p.cam_pos[0], p.cam_pos[1], p.cam_pos[2]), v3(p.look_at[0], p.look_at[1], p.look_at[2]),
                        p.vfov, p.aperture, p.focus_dist, p.width, p.height);
}

// render.rs:163-182 — the primary ray of (pixel idx, sample s).
static Ray primary_ray(const RenderParams& p, const Camera& cam, size_t idx, uint32_t s, Rng& rng) {
    size_t px = idx % p.width;                // util.rs:31-33  Coord::from_index
    size_t py = p.height - (idx / p.width);
    rng.begin((uint32_t)idx, s);
    rng.set_stream(0, STREAM_CAMERA);
    float u = ((float)px + rng.rand_f32()) / (float)p.width;
    float v = ((float)py + rng.rand_f32()) / (float)p.height;
    return cam.ray(u, v, rng);
}

// util.rs:14-23 + render.rs:184-189
static void resolve_pixel(Vec3 total, uint32_t samples, float gamma, uint8_t out[3]) {
    total = total / (float)samples;
    float g = 1.0f / gamma;
    float c[3] = {total.x, total.y, total.z};
    for (int k = 0; k < 3; ++k) {
        float x = std::pow(c[k], g);
        // f32::clamp(0,1): NaN stays NaN
        if (x < 0.0f) x = 0.0f;
        if (x > 1.0f) x = 1.0f;
        out[k] = f32_as_u8(x * 255.99f);
    }
}

}  // namespace orc

// =================================================================================================
// C ABI for the ctypes harness (oracle/oracle.py).  Builder-style: the harness parses the serde YAML
// with PyYAML and replays it through these calls.
// =================================================================================================
using namespace orc;

// Flattened description of a BVH for structural tests: pre-order list of
// {kind, item_a, item_b, min[3], max[3]} as 9 floats... kept simple: returns node count & leaf order.
template <class T, class F>
static void bvh_walk(const BVHNode<T>* n, F&& f, int depth) {
    f(n, depth);
    if (n->kind == BVHNode<T>::BRANCH) {
        bvh_walk<T>(n->l.get(), f, depth + 1);
        bvh_walk<T>(n->r.get(), f, depth + 1);
    }
}
extern "C" {

void* orc_scene_new() { return new Scene(); }
void orc_scene_free(void* s) { delete (Scene*)s; }

int orc_tex_constant(void* sp, float r, float g, float b) {
    Scene* s = (Scene*)sp;
    auto t = std::make_unique<ConstantTexture>();
    t->color = v3(r, g, b);
    s->textures.push_back(std::move(t));
    return (int)s->textures.size() - 1;
}
int orc_tex_checker(void* sp, int odd, int even, float scale) {
    Scene* s = (Scene*)sp;
    auto t = std::make_unique<CheckerTexture>();
    t->odd = s->textures.at(odd).get();
    t->even = s->textures.at(even).get();
    t->scale = scale;
    s->textures.push_back(std::move(t));
    return (int)s->textures.size() - 1;
}
int orc_tex_perlin(void* sp, float scale) {
    Scene* s = (Scene*)sp;
    auto t = std::make_unique<PerlinNoiseTexture>();
    t->scale = scale;
    s->textures.push_back(std::move(t));
    return (int)s->textures.size() - 1;
}
int orc_tex_turbulence(void* sp, uint64_t depth, float scale) {
    Scene* s = (Scene*)sp;
    auto t = std::make_unique<TurbulenceTexture>();
    t->depth = depth;
    t->scale = scale;
    s->textures.push_back(std::move(t));
    return (int)s->textures.size() - 1;
}
int orc_tex_marble(void* sp, uint64_t depth, float scale) {
    Scene* s = (Scene*)sp;
    auto t = std::make_unique<MarbleTexture>();
    t->depth = depth;
    t->scale = scale;
    s->textures.push_back(std::move(t));
    return (int)s->textures.size() - 1;
}
int orc_tex_image(void* sp, uint32_t w, uint32_t h, const uint8_t* rgba) {
    Scene* s = (Scene*)sp;
    auto t = std::make_unique<ImageTexture>();
    t->w = w;
    t->h = h;
    t->rgba.assign(rgba, rgba + (size_t)w * h * 4);
    s->textures.push_back(std::move(t));
    return (int)s->textures.size() - 1;
}

// kind: 0 Lambertian(tex) 1 Metal(albedo, roughness) 2 Dielectric(ref_idx) 3 Emissive(tex) 4 Isotropic(tex)
int orc_material(void* sp, int kind, int tex, const float albedo[3], float param) {
    Scene* s = (Scene*)sp;
    std::unique_ptr<Material> m;
    switch (kind) {
        case 0: { auto x = std::make_unique<LambertianMat>(); x->albedo = s->textures.at(tex).get(); m = std::move(x); break; }
        case 1: { auto x = std::make_unique<MetalMat>(); x->albedo = v3(albedo[0], albedo[1], albedo[2]); x->roughness = param; m = std::move(x); break; }
        case 2: { auto x = std::make_unique<DielectricMat>(); x->ref_idx = param; m = std::move(x); break; }
        case 3: { auto x = std::make_unique<EmissiveMat>(); x->albedo = s->textures.at(tex).get(); m = std::move(x); break; }
        case 4: { auto x = std::make_unique<IsotropicMat>(); x->texture = s->textures.at(tex).get(); m = std::move(x); break; }
        default: return -1;
    }
    s->materials.push_back(std::move(m));
    s->material_kind.push_back(kind);
    return (int)s->materials.size() - 1;
}

static int push_shape(Scene* s, std::unique_ptr<Hitable> h) {
    s->shapes.push_back(std::move(h));
    return (int)s->shapes.size() - 1;
}
int orc_shape_sphere(void* sp, float radius, int material) {
    auto x = std::make_unique<Sphere>();
    x->radius = radius;
    x->material = material;
    return push_shape((Scene*)sp, std::move(x));
}
static void fill_rect(AARect& x, int plane, const float mn[2], const float mx[2], float k, int flip, int material) {
    static const int A1[3] = {0, 0, 1}, A2[3] = {1, 2, 2}, AK[3] = {2, 1, 0};  // XY, XZ, YZ
    x.a1 = A1[plane]; x.a2 = A2[plane]; x.ak = AK[plane];
    x.min = Vec2{mn[0], mn[1]};
    x.max = Vec2{mx[0], mx[1]};
    x.k = k;
    x.flip_normal = flip != 0;
    x.material = material;
}
// plane: 0 = XY, 1 = XZ, 2 = YZ
int orc_shape_rect(void* sp, int plane, const float mn[2], const float mx[2], float k, int flip, int material) {
    auto x = std::make_unique<AARect>();
    fill_rect(*x, plane, mn, mx, k, flip, material);
    return push_shape((Scene*)sp, std::move(x));
}
// faces: nfaces × {plane, min.x, min.y, max.x, max.y, k, flip, material} as 8 floats each
int orc_shape_rect3d(void* sp, const float pos[3], const float size[3], int nfaces, const float* faces) {
    auto x = std::make_unique<Rect3d>();
    x->pos = v3(pos[0], pos[1], pos[2]);
    x->size = v3(size[0], size[1], size[2]);
    for (int i = 0; i < nfaces; ++i) {
        const float* f = faces + 8 * i;
        AARect r;
        float mn[2] = {f[1], f[2]}, mx[2] = {f[3], f[4]};
        fill_rect(r, (int)f[0], mn, mx, f[5], (int)f[6], (int)f[7]);
        x->faces.push_back(r);
    }
    return push_shape((Scene*)sp, std::move(x));
}
int orc_shape_disk(void* sp, float radius, float phi_max, float inner_radius, int material) {
    auto x = std::make_unique<Disk>();
    x->radius = radius; x->phi_max = phi_max; x->inner_radius = inner_radius; x->material = material;
    return push_shape((Scene*)sp, std::move(x));
}
int orc_shape_cylinder(void* sp, float radius, float height, float max_phi, int material) {
    auto x = std::make_unique<Cylinder>();
    x->radius = radius; x->height = height; x->max_phi = max_phi; x->material = material;
    return push_shape((Scene*)sp, std::move(x));
}
int orc_shape_cone(void* sp, float radius, float height, int material) {
    auto x = std::make_unique<Cone>();
    x->radius = radius; x->height = height; x->material = material;
    return push_shape((Scene*)sp, std::move(x));
}
int orc_shape_mesh(void* sp, uint32_t nverts, const float* verts, uint32_t nidx, const uint32_t* idx,
                   const float* normals, const float* uvs, int material) {
    Scene* s = (Scene*)sp;
    auto m = std::make_shared<TriangleMesh>();
    m->verts.resize(nverts);
    for (uint32_t i = 0; i < nverts; ++i) m->verts[i] = v3(verts[3 * i], verts[3 * i + 1], verts[3 * i + 2]);
    m->indicies.assign(idx, idx + nidx);
    if (normals) {
        m->has_normals = true;
        m->normals.resize(nverts);
        for (uint32_t i = 0; i < nverts; ++i) m->normals[i] = v3(normals[3 * i], normals[3 * i + 1], normals[3 * i + 2]);
    }
    if (uvs) {
        m->has_uvs = true;
        m->uvs.resize(nverts);
        for (uint32_t i = 0; i < nverts; ++i) m->uvs[i] = Vec2{uvs[2 * i], uvs[2 * i + 1]};
    }
    m->material = material;
    s->meshes.push_back(m);
    auto x = std::make_unique<MeshBVH>();
    x->mesh = m;
    x->build();
    return push_shape(s, std::move(x));
}
int orc_shape_medium(void* sp, int inner_shape, float density, int material) {
    Scene* s = (Scene*)sp;
    auto x = std::make_unique<ConstantMedium>();
    x->obj = std::move(s->shapes.at(inner_shape));
    if (!x->obj) return -1;
    x->density = density;
    x->material = material;
    return push_shape(s, std::move(x));
}
// rotor = {s, xy, xz, yz}
int orc_add_object(void* sp, int shape, const float pos[3], const float rotor[4], int flip_normals) {
    Scene* s = (Scene*)sp;
    auto ro = std::make_unique<RenderObjectInternal>();
    ro->obj = std::move(s->shapes.at(shape));
    if (!ro->obj) return -1;
    ro->position = v3(pos[0], pos[1], pos[2]);
    Rotor3 r{rotor[0], rotor[1], rotor[2], rotor[3]};
    ro->rotation_mat = rotor_into_matrix(r);                      // scene.rs:284
    ro->inv_rotation_mat = rotor_into_matrix(rotor_reversed(r));  // scene.rs:285
    ro->flip_normals = flip_normals != 0;
    ro->id = (int)s->render_objects.size();
    if (auto* med = dynamic_cast<ConstantMedium*>(ro->obj.get())) med->rng_id = ro->id;
    ro->update_bounding_box();
    s->render_objects.push_back(std::move(ro));
    return (int)s->render_objects.size() - 1;
}
void orc_env_color(void* sp, float r, float g, float b) {
    auto e = std::make_unique<ColorEnv>();
    e->color = v3(r, g, b);
    ((Scene*)sp)->environment = std::move(e);
}
void orc_env_sky(void* sp, const float zenith[3], const float horizon[3]) {
    auto e = std::make_unique<SkyEnv>();
    e->zenith_color = v3(zenith[0], zenith[1], zenith[2]);
    e->horizon_color = v3(horizon[0], horizon[1], horizon[2]);
    ((Scene*)sp)->environment = std::move(e);
}
void orc_env_hdr(void* sp, uint32_t w, uint32_t h, const float* rgb) {
    auto e = std::make_unique<HdrEnvironment>();
    e->pixels.assign(rgb, rgb + (size_t)w * h * 3);
    e->width = (float)w;
    e->height = (float)h;
    ((Scene*)sp)->environment = std::move(e);
}
// Finish: default environment (scene.rs:36: black ColorEnv) and the optional top-level BVH.
int orc_scene_finish(void* sp, int build_bvh) {
    Scene* s = (Scene*)sp;
    if (!s->environment) orc_env_color(sp, 0, 0, 0);
    if (s->render_objects.empty()) return -1;
    if (build_bvh) s->build_bvh();
    return 0;
}

int orc_num_objects(void* sp) { return (int)((Scene*)sp)->render_objects.size(); }
void orc_object_aabb(void* sp, int i, float out[6]) {
    const AABB& b = ((Scene*)sp)->render_objects.at(i)->aabb;
    out[0] = b.min.x; out[1] = b.min.y; out[2] = b.min.z; out[3] = b.max.x; out[4] = b.max.y; out[5] = b.max.z;
}
void orc_object_rotation(void* sp, int i, float out[9]) {
    const Mat3& m = ((Scene*)sp)->render_objects.at(i)->rotation_mat;
    for (int c = 0; c < 3; ++c) { out[3 * c] = m.cols[c].x; out[3 * c + 1] = m.cols[c].y; out[3 * c + 2] = m.cols[c].z; }
}

// Leaf order (DFS) of the top-level BVH: writes object ids, returns count; out may be null.
int orc_bvh_leaf_order(void* sp, int* out, int cap, int* n_nodes, int* max_depth) {
    Scene* s = (Scene*)sp;
    if (!s->bvh) return -1;
    int cnt = 0, nodes = 0, md = 0;
    bvh_walk<const RenderObjectInternal*>(s->bvh.get(), [&](const BVHNode<const RenderObjectInternal*>* n, int d) {
        ++nodes;
        md = std::max(md, d);
        if (n->kind == BVHNode<const RenderObjectInternal*>::LEAF) {
            if (out && cnt < cap) out[cnt] = n->a->id;
            ++cnt;
        } else if (n->kind == BVHNode<const RenderObjectInternal*>::DOUBLE_LEAF) {
            if (out && cnt < cap) out[cnt] = n->a->id;
            ++cnt;
            if (out && cnt < cap) out[cnt] = n->b->id;
            ++cnt;
        }
    }, 0);
    if (n_nodes) *n_nodes = nodes;
    if (max_depth) *max_depth = md;
    return cnt;
}
// Pre-order dump of the top-level BVH boxes: 7 floats per node {kind, min3, max3}.
int orc_bvh_nodes(void* sp, float* out, int cap_nodes) {
    Scene* s = (Scene*)sp;
    if (!s->bvh) return -1;
    int nodes = 0;
    bvh_walk<const RenderObjectInternal*>(s->bvh.get(), [&](const BVHNode<const RenderObjectInternal*>* n, int) {
        if (out && nodes < cap_nodes) {
            float* o = out + 7 * nodes;
            o[0] = (float)n->kind;
            o[1] = n->aabb.min.x; o[2] = n->aabb.min.y; o[3] = n->aabb.min.z;
            o[4] = n->aabb.max.x; o[5] = n->aabb.max.y; o[6] = n->aabb.max.z;
        }
        ++nodes;
    }, 0);
    return nodes;
}
// Leaf order of mesh object i's triangle BVH (object must be a TriangleMesh).
int orc_mesh_leaf_order(void* sp, int obj, int* out, int cap, int* n_nodes, int* max_depth) {
    Scene* s = (Scene*)sp;
    auto* mb = dynamic_cast<MeshBVH*>(s->render_objects.at(obj)->obj.get());
    if (!mb) return -1;
    int cnt = 0, nodes = 0, md = 0;
    bvh_walk<Triangle>(mb->root.get(), [&](const BVHNode<Triangle>* n, int d) {
        ++nodes;
        md = std::max(md, d);
        if (n->kind == BVHNode<Triangle>::LEAF) {
            if (out && cnt < cap) out[cnt] = (int)n->a.index;
            ++cnt;
        } else if (n->kind == BVHNode<Triangle>::DOUBLE_LEAF) {
            if (out && cnt < cap) out[cnt] = (int)n->a.index;
            ++cnt;
            if (out && cnt < cap) out[cnt] = (int)n->b.index;
            ++cnt;
        }
    }, 0);
    if (n_nodes) *n_nodes = nodes;
    if (max_depth) *max_depth = md;
    return cnt;
}

struct OrcStats {
    uint64_t samples, rays, aabb_tests, prim_tests;
    double seconds;
    int threads;
    int pad;
    uint64_t sphere, rect, tri, conic, xform_rot, xform_trans;
};

// The camera (camera.rs:74-107) as 8 Vec3-ish constants: position, horizontal, vertical, lower_left, u, v, w,
// (lens_radius, 0, 0) -> 24 floats.
void orc_camera(const RenderParams* p, float out[24]) {
    Camera c = make_camera(*p);
    const Vec3 vs[7] = {c.position, c.horizontal, c.vertical, c.lower_left, c.u, c.v, c.w};
    for (int i = 0; i < 7; ++i) { out[3 * i] = vs[i].x; out[3 * i + 1] = vs[i].y; out[3 * i + 2] = vs[i].z; }
    out[21] = c.lens_radius; out[22] = 0; out[23] = 0;
}

// Primary rays of sample index `s` for pixels [pix_begin, pix_begin+n): origins/dirs n×3.
void orc_primary_rays(const RenderParams* p, uint32_t s, uint32_t pix_begin, uint32_t n, float* origins, float* dirs) {
    Camera cam = make_camera(*p);
#pragma omp parallel for schedule(static)
    for (int64_t i = 0; i < (int64_t)n; ++i) {
        Rng rng;
        rng.seed(p->seed);
        Ray r = primary_ray(*p, cam, pix_begin + (size_t)i, s, rng);
        origins[3 * i] = r.origin.x; origins[3 * i + 1] = r.origin.y; origins[3 * i + 2] = r.origin.z;
        dirs[3 * i] = r.dir.x; dirs[3 * i + 1] = r.dir.y; dirs[3 * i + 2] = r.dir.z;
    }
}

// Closest-hit probe (render.rs:19): rays with their RNG keys (pixel, sample, bounce) -> hit records.
// obj_id = -1 on miss.
void orc_first_hit(void* sp, int use_bvh, uint64_t seed, uint32_t n, const float* origins, const float* dirs,
                   const uint32_t* pixel, const uint32_t* sample, const uint32_t* bounce, int32_t* obj_id,
                   int32_t* prim_id, int32_t* material, float* t, float* point, float* normal, float* uv,
                   OrcStats* stats) {
    Scene* s = (Scene*)sp;
    uint64_t aabb = 0, prim = 0;
#pragma omp parallel for schedule(dynamic, 256) reduction(+ : aabb, prim)
    for (int64_t i = 0; i < (int64_t)n; ++i) {
        g_cnt = Counters();
        Rng rng;
        rng.seed(seed);
        rng.begin(pixel ? pixel[i] : (uint32_t)i, sample ? sample[i] : 0);
        rng.set_stream(bounce ? bounce[i] : 0, STREAM_MEDIUM);
        Ray r{v3(origins[3 * i], origins[3 * i + 1], origins[3 * i + 2]), v3(dirs[3 * i], dirs[3 * i + 1], dirs[3 * i + 2])};
        RaycastHit h;
        bool ok = s->root_hit(use_bvh != 0, r, 0.001f, 2e9f, rng, h);
        if (ok) {
            obj_id[i] = h.obj_id; prim_id[i] = h.prim_id; material[i] = h.material; t[i] = h.t;
            point[3 * i] = h.point.x; point[3 * i + 1] = h.point.y; point[3 * i + 2] = h.point.z;
            normal[3 * i] = h.normal.x; normal[3 * i + 1] = h.normal.y; normal[3 * i + 2] = h.normal.z;
            uv[2 * i] = h.uv.x; uv[2 * i + 1] = h.uv.y;
        } else {
            obj_id[i] = -1; prim_id[i] = 0; material[i] = -1; t[i] = 0;
            point[3 * i] = point[3 * i + 1] = point[3 * i + 2] = 0;
            normal[3 * i] = normal[3 * i + 1] = normal[3 * i + 2] = 0;
            uv[2 * i] = uv[2 * i + 1] = 0;
        }
        aabb += g_cnt.aabb_tests;
        prim += g_cnt.prim_tests;
    }
    if (stats) { stats->rays = n; stats->aabb_tests = aabb; stats->prim_tests = prim; stats->samples = 0; }
}

// One scatter step (render.rs:20-22) of item i:
// in:  material id, ray (o,d), hit (t, point, normal, uv), the item's random stream
// out: emit[3], scattered flag, attenuation[3], new ray o[3], d[3]
static void scatter_one(Scene* s, uint32_t i, const int32_t* material, const float* ray_o, const float* ray_d,
                        const float* hit_t, const float* hit_point, const float* hit_normal, const float* hit_uv, Rng& rng,
                        float* emit, int32_t* scattered, float* atten, float* out_o, float* out_d) {
    Ray r{v3(ray_o[3 * i], ray_o[3 * i + 1], ray_o[3 * i + 2]), v3(ray_d[3 * i], ray_d[3 * i + 1], ray_d[3 * i + 2])};
    RaycastHit h;
    h.t = hit_t[i];
    h.point = v3(hit_point[3 * i], hit_point[3 * i + 1], hit_point[3 * i + 2]);
    h.normal = v3(hit_normal[3 * i], hit_normal[3 * i + 1], hit_normal[3 * i + 2]);
    h.uv = Vec2{hit_uv[2 * i], hit_uv[2 * i + 1]};
    h.material = material[i];
    const Material& m = *s->materials.at(material[i]);
    Vec3 e = m.emit(h.uv, h.point);
    ScatterResult res;
    res.attenuation = v3(0, 0, 0);
    res.scattered = Ray{v3(0, 0, 0), v3(0, 0, 0)};
    bool ok = m.scatter(r, h, rng, res);
    emit[3 * i] = e.x; emit[3 * i + 1] = e.y; emit[3 * i + 2] = e.z;
    scattered[i] = ok ? 1 : 0;
    if (!ok) { res.attenuation = v3(0, 0, 0); res.scattered = Ray{v3(0, 0, 0), v3(0, 0, 0)}; }
    atten[3 * i] = res.attenuation.x; atten[3 * i + 1] = res.attenuation.y; atten[3 * i + 2] = res.attenuation.z;
    out_o[3 * i] = res.scattered.origin.x; out_o[3 * i + 1] = res.scattered.origin.y; out_o[3 * i + 2] = res.scattered.origin.z;
    out_d[3 * i] = res.scattered.dir.x; out_d[3 * i + 1] = res.scattered.dir.y; out_d[3 * i + 2] = res.scattered.dir.z;
}
// ... with EXPLICIT uniforms consumed in order (nu per item); consumed = uniforms used, -1 on overrun
void orc_scatter_step(void* sp, uint32_t n, const int32_t* material, const float* ray_o, const float* ray_d,
                      const float* hit_t, const float* hit_point, const float* hit_normal, const float* hit_uv,
                      const float* uniforms, uint32_t nu, float* emit, int32_t* scattered, float* atten,
                      float* out_o, float* out_d, int32_t* consumed) {
    Scene* s = (Scene*)sp;
    for (uint32_t i = 0; i < n; ++i) {
        Rng rng;
        rng.arr = uniforms + (size_t)i * nu;
        rng.arr_n = (int)nu;
        scatter_one(s, i, material, ray_o, ray_d, hit_t, hit_point, hit_normal, hit_uv, rng, emit, scattered, atten, out_o, out_d);
        consumed[i] = rng.arr_overrun ? -1 : rng.arr_i;
    }
}
// ... drawing from the keyed stream color() uses at bounce[i] of (pixel[i], sample[i]); consumed = uniforms drawn
void orc_scatter_step_keyed(void* sp, uint64_t seed, uint32_t n, const int32_t* material, const float* ray_o,
                            const float* ray_d, const float* hit_t, const float* hit_point, const float* hit_normal,
                            const float* hit_uv, const uint32_t* pixel, const uint32_t* sample, const uint32_t* bounce,
                            float* emit, int32_t* scattered, float* atten, float* out_o, float* out_d, int32_t* consumed) {
    Scene* s = (Scene*)sp;
    for (uint32_t i = 0; i < n; ++i) {
        Rng rng;
        rng.seed(seed);
        rng.begin(pixel[i], sample[i]);
        rng.set_stream(bounce[i], STREAM_SCATTER);
        scatter_one(s, i, material, ray_o, ray_d, hit_t, hit_point, hit_normal, hit_uv, rng, emit, scattered, atten, out_o, out_d);
        consumed[i] = (int32_t)rng.idx;
    }
}

// Environment lookup probe (render.rs:31): dirs are normalised by the caller exactly as color() does.
void orc_env_sample(void* sp, uint32_t n, const float* dirs, float* out) {
    Scene* s = (Scene*)sp;
    for (uint32_t i = 0; i < n; ++i) {
        Vec3 d = normalized(v3(dirs[3 * i], dirs[3 * i + 1], dirs[3 * i + 2]));
        Vec3 c = s->environment->sample(d);
        out[3 * i] = c.x; out[3 * i + 1] = c.y; out[3 * i + 2] = c.z;
    }
}
// Texture lookup probe.
void orc_texture_sample(void* sp, int tex, uint32_t n, const float* uv, const float* point, float* out) {
    Scene* s = (Scene*)sp;
    const Texture& t = *s->textures.at(tex);
    for (uint32_t i = 0; i < n; ++i) {
        Vec3 c = t.sample(Vec2{uv[2 * i], uv[2 * i + 1]}, v3(point[3 * i], point[3 * i + 1], point[3 * i + 2]));
        out[3 * i] = c.x; out[3 * i + 1] = c.y; out[3 * i + 2] = c.z;
    }
}
float orc_perlin_noise(float x, float y, float z) { return perlin_noise(v3(x, y, z)); }

// Renderer::render (render.rs:109-196) for samples [sample_begin, sample_begin+sample_count):
//   sum_out  (nullable) : width*height*3 fp32 un-normalised sums, accumulated in sample order
//   rgb_out  (nullable) : width*height*3 u8, = resolve(sum / samples)   (only meaningful when the call
//                         covers the whole sample range)
// pix_begin/pix_count restrict the pixel range (row-major idx) — used by the bounded CPU baseline.
int orc_render(void* sp, const RenderParams* p, uint32_t pix_begin, uint32_t pix_count, float* sum_out,
               uint8_t* rgb_out, OrcStats* stats, int num_threads) {
    Scene* s = (Scene*)sp;
    if (p->use_bvh && !s->bvh) return -2;
    Camera cam = make_camera(*p);
    uint64_t rays = 0, aabb = 0, prim = 0, k_sph = 0, k_rect = 0, k_tri = 0, k_con = 0, k_xr = 0, k_xt = 0;
    int threads = 1;
#ifdef _OPENMP
    if (num_threads > 0) omp_set_num_threads(num_threads);
    threads = omp_get_max_threads();
    double t0 = omp_get_wtime();
#else
    double t0 = 0;
#endif
    if (pix_count == 0) pix_count = p->width * p->height - pix_begin;
    // render.rs:127 — one task per pixel (rayon work stealing ~ schedule(dynamic))
#pragma omp parallel for schedule(dynamic, 16) reduction(+ : rays, aabb, prim, k_sph, k_rect, k_tri, k_con, k_xr, k_xt)
    for (int64_t k = 0; k < (int64_t)pix_count; ++k) {
        size_t idx = pix_begin + (size_t)k;
        g_cnt = Counters();
        Rng rng;
        rng.seed(p->seed);
        Vec3 total = v3(0, 0, 0);
        for (uint32_t si = 0; si < p->sample_count; ++si) {  // render.rs:177-182
            uint32_t smp = p->sample_begin + si;
            Ray ray = primary_ray(*p, cam, idx, smp, rng);
            total = total + color(ray, *s, p->use_bvh != 0, 0, rng);
        }
        if (sum_out) { sum_out[3 * idx] = total.x; sum_out[3 * idx + 1] = total.y; sum_out[3 * idx + 2] = total.z; }
        if (rgb_out) resolve_pixel(total, p->samples, p->gamma, rgb_out + 3 * idx);
        rays += g_cnt.rays; aabb += g_cnt.aabb_tests; prim += g_cnt.prim_tests;
        k_sph += g_cnt.sphere; k_rect += g_cnt.rect; k_tri += g_cnt.tri; k_con += g_cnt.conic;
        k_xr += g_cnt.xform_rot; k_xt += g_cnt.xform_trans;
    }
    if (stats) {
        stats->samples = (uint64_t)pix_count * p->sample_count;
        stats->rays = rays; stats->aabb_tests = aabb; stats->prim_tests = prim;
        stats->sphere = k_sph; stats->rect = k_rect; stats->tri = k_tri; stats->conic = k_con;
        stats->xform_rot = k_xr; stats->xform_trans = k_xt;
#ifdef _OPENMP
        stats->seconds = omp_get_wtime() - t0;
#else
        stats->seconds = 0;
#endif
        stats->threads = threads;
    }
    return 0;
}

// resolve only (render.rs:184-189 + util.rs:14-23) from an fp32 sum buffer.
void orc_resolve(const float* sum, uint32_t npix, uint32_t samples, float gamma, uint8_t* rgb) {
    for (uint32_t i = 0; i < npix; ++i) resolve_pixel(v3(sum[3 * i], sum[3 * i + 1], sum[3 * i + 2]), samples, gamma, rgb + 3 * i);
}

// Philox known-answer access for tests.
void orc_philox(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]) { philox4x32_10(ctr, key, out); }

}  // extern "C"
