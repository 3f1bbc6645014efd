// Material scatter / emit, texture and environment lookups: the CUDA counterparts of
//   material.rs:65-74 (Lambertian), 91-106 (Metal), 122-150 (Dielectric), 174-180 (Emissive), 198-203 (Isotropic)
//   util.rs:36-73 (rejection samplers, reflect, refract, schlick)
//   texture.rs:31-33, 59-72, 113-193, 206-224, 241-248, 296-309
//   environment.rs:23-25, 62-66 and examples/hdri_test.rs:14-20, 72-81
// Operation order follows the reference; see device_math.cuh for the arithmetic-fidelity rules.
#pragma once
#include "device_math.cuh"
#include "fw_types.h"

namespace fw {

// texture.rs:82-106 — Ken Perlin's reference permutation (published constant); P[512] = P256 ++ P256.
__device__ const unsigned char FW_PERLIN_P[256] = {
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
FW_DEV unsigned perlin_p(unsigned i) { return FW_PERLIN_P[i & 255u]; }

FW_DEV float perlin_fade(float t) { return t * t * (3.0f - 2.0f * t); }  // texture.rs:163-166
FW_DEV float perlin_grad(unsigned hash, float x, float y, float z) {      // texture.rs:168-182
    unsigned h = hash & 15u;
    float u = h < 8u ? x : y;
    float v = h < 4u ? y : ((h == 12u || h == 14u) ? x : z);
    u = (h & 1u) == 0u ? u : -u;
    v = (h & 2u) == 0u ? v : -v;
    return u + v;
}
FW_DEV float perlin_lerp(float t, float a, float b) { return a + t * (b - a); }  // texture.rs:184-186
// `floor(x) as usize & 255`: the Rust cast saturates (negatives and NaN -> 0, huge -> usize::MAX -> 255)
FW_DEV unsigned perlin_cell(float f) { return (unsigned)(__float2ull_rz(f) & 255ull); }
// Rust `f as u64` / `f as u32`: saturating, NaN -> 0.  The hardware conversion saturates but does not map NaN to 0.
FW_DEV unsigned long long f32_as_u64(float f) { return f == f ? __float2ull_rz(f) : 0ull; }
FW_DEV uint32_t f32_as_u32(float f) { return f == f ? __float2uint_rz(f) : 0u; }
FW_DEV float perlin_noise(float3 p) {  // texture.rs:113-158
    float fx = floorf(p.x), fy = floorf(p.y), fz = floorf(p.z);
    unsigned x0 = perlin_cell(fx), y0 = perlin_cell(fy), z0 = perlin_cell(fz);
    float x = p.x - fx, y = p.y - fy, z = p.z - fz;
    float u = perlin_fade(x), v = perlin_fade(y), w = perlin_fade(z);
    unsigned a = perlin_p(x0) + y0;
    unsigned aa = perlin_p(a) + z0;
    unsigned ab = perlin_p(a + 1) + z0;
    unsigned b = perlin_p(x0 + 1) + y0;
    unsigned ba = perlin_p(b) + z0;
    unsigned bb = perlin_p(b + 1) + z0;
    return perlin_lerp(
        w,
        perlin_lerp(v, perlin_lerp(u, perlin_grad(perlin_p(aa), x, y, z), perlin_grad(perlin_p(ba), x - 1.0f, y, z)),
                    perlin_lerp(u, perlin_grad(perlin_p(ab), x, y - 1.0f, z),
                                perlin_grad(perlin_p(bb), x - 1.0f, y - 1.0f, z))),
        perlin_lerp(v,
                    perlin_lerp(u, perlin_grad(perlin_p(aa + 1), x, y, z - 1.0f),
                                perlin_grad(perlin_p(ba + 1), x - 1.0f, y, z - 1.0f)),
                    perlin_lerp(u, perlin_grad(perlin_p(ab + 1), x, y - 1.0f, z - 1.0f),
                                perlin_grad(perlin_p(bb + 1), x - 1.0f, y - 1.0f, z - 1.0f))));
}
FW_DEV float turbulence(int depth, float3 point) {  // texture.rs:206-217 — no abs()
    float accum = 0.0f;
    float3 p = point;
    float weight = 1.0f;
    for (int i = 0; i < depth; ++i) {
        float a = perlin_noise(p);
        accum += weight * a;
        weight *= 0.5f;
        p = p * 2.0f;
    }
    return accum;
}

FW_DEV float3 texture_sample(const DeviceScene& S, int tex, float2 uv, float3 point) {
    for (int guard = 0; guard < FW_MAX_TEXTURE_DEPTH; ++guard) {
        const float4* q = reinterpret_cast<const float4*>(&S.texs[tex]);
        float4 q0 = __ldg(q), q1 = __ldg(q + 1);
        int kind = __float_as_int(q0.x);
        float scale = q1.x;
        switch (kind) {
            case TEX_CONSTANT:  // texture.rs:31-33
                return f3(q1.y, q1.z, q1.w);
            case TEX_CHECKER: {  // texture.rs:59-72 — product().is_sign_positive()
                float ax = scale * point.x, ay = scale * point.y, az = scale * point.z;
                float prod = 1.0f;
                prod = prod * sinf(ax);
                prod = prod * sinf(ay);
                prod = prod * sinf(az);
                bool odd = signbit(prod);
                if (prod != prod) {
                    // The reference's NaN sign is x86's (DESIGN.md §3): the first axis whose sin is NaN decides; that NaN is
                    // the coordinate's own, or the negative default NaN of sin(±inf) / 0 * inf.  Device arithmetic yields
                    // only the positive canonical NaN, so the sign is decided here.
                    float c = isfinite(ax) ? (isfinite(ay) ? point.z : point.y) : point.x;
                    odd = !(c != c) || signbit(c);
                }
                tex = odd ? __float_as_int(q0.y) : __float_as_int(q0.z);  // odd : even
                continue;
            }
            case TEX_PERLIN: {  // texture.rs:160-167
                float a = perlin_noise(point * scale);
                float v = fminf(a + 0.5f, 1.0f);
                return f3(1.0f * v, 1.0f * v, 1.0f * v);
            }
            case TEX_TURBULENCE: {  // texture.rs:219-224
                float v = turbulence(__float_as_int(q0.w), point * scale);
                return f3(1.0f * v, 1.0f * v, 1.0f * v);
            }
            case TEX_MARBLE: {  // texture.rs:241-248
                float v = 0.5f * (1.0f + sinf(scale * point.z + 10.0f * turbulence(__float_as_int(q0.w), point)));
                return f3(v, v, v);
            }
            case TEX_IMAGE: {  // texture.rs:296-309 — nearest texel, v flipped, clamp to edge
                const ImageRec* im = &S.images[__float_as_int(q0.y)];
                uint32_t w = im->w, h = im->h;
                float fi = uv.x * (float)w;
                float fj = (1.0f - uv.y) * (float)h;
                uint32_t i = min(f32_as_u32(fi), w - 1);
                uint32_t j = min(f32_as_u32(fj), h - 1);
                uchar4 c = tex2D<uchar4>(im->tex, (float)i + 0.5f, (float)j + 0.5f);
                return f3((float)c.x, (float)c.y, (float)c.z) / 255.0f;
            }
            default:
                return f3(0.0f, 0.0f, 0.0f);
        }
    }
    return f3(0.0f, 0.0f, 0.0f);
}

// environment.rs:23-25, 62-66; hdri_test.rs:72-81.  `dir` is the ray direction; color() normalises it
// (render.rs:31).
FW_DEV float3 environment_sample(const EnvRec& env, float3 raw_dir) {
    float3 dir = normalized3(raw_dir);
    if (env.kind == ENV_COLOR) return f3(env.a[0], env.a[1], env.a[2]);
    if (env.kind == ENV_SKY) {
        float t = 0.5f * (dir.y + 1.0f);
        float3 horizon = f3(env.b[0], env.b[1], env.b[2]), zenith = f3(env.a[0], env.a[1], env.a[2]);
        return (1.0f - t) * horizon + t * zenith;
    }
    // equirectangular nearest lookup
    float phi = atan2f(dir.z, dir.x);
    float theta = asinf(dir.y);
    float u = 1.0f - (phi + FW_PI) / (2.0f * FW_PI);
    float v = (theta + FW_PI / 2.0f) / FW_PI;
    float width = (float)env.w, height = (float)env.h;
    unsigned long long x = f32_as_u64(u * width);
    unsigned long long y = f32_as_u64((1.0f - v) * height);
    unsigned long long idx = f32_as_u64((float)y * width) + x;
    // DEVIATION (documented in DESIGN.md): the reference panics on an out-of-range index (dir.y == -1);
    // here the index is clamped to the last texel.
    unsigned long long n = (unsigned long long)env.w * env.h;
    if (idx >= n) idx = n - 1;
    uint32_t yy = (uint32_t)(idx / env.w), xx = (uint32_t)(idx % env.w);
    float4 c = tex2D<float4>(env.tex, (float)xx + 0.5f, (float)yy + 0.5f);
    return f3(c.x, c.y, c.z);
}

// util.rs:36-43
template <class Stream>
FW_DEV float3 random_in_unit_sphere(Stream& rng) {
    for (;;) {
        float a = rng.next(), b = rng.next(), c = rng.next();
        float3 p = 2.0f * f3(a, b, c) - f3(1.0f, 1.0f, 1.0f);
        if (mag_sq3(p) < 1.0f) return p;
    }
}
// The same sampler for a FRESH Philox stream (idx == 0), restructured for SIMT: the rejection loop makes a warp
// wait for its unluckiest lane (mean 1.9 rounds, max over 32 lanes ~6), so the first four rounds (12 uniforms =
// 3 Philox blocks) are generated unconditionally and the first accepted one is picked without branching; only
// lanes that fail four times (4.9 %) fall back to the sequential loop.  Consumes exactly the same uniforms in
// the same order as the loop above, so the result is identical.
FW_DEV float3 random_in_unit_sphere_fresh(PhiloxStream& rng) {
    uint32_t w1 = (rng.key.bounce << 8) | rng.kind;
    uint4 b0 = philox4x32_10(make_uint4(0u, w1, rng.key.sample, rng.key.pixel), rng.key.seed);
    uint4 b1 = philox4x32_10(make_uint4(1u, w1, rng.key.sample, rng.key.pixel), rng.key.seed);
    uint4 b2 = philox4x32_10(make_uint4(2u, w1, rng.key.sample, rng.key.pixel), rng.key.seed);
    const float3 one = f3(1.0f, 1.0f, 1.0f);
    float3 p0 = 2.0f * f3(u32_to_unit(b0.x), u32_to_unit(b0.y), u32_to_unit(b0.z)) - one;
    float3 p1 = 2.0f * f3(u32_to_unit(b0.w), u32_to_unit(b1.x), u32_to_unit(b1.y)) - one;
    float3 p2 = 2.0f * f3(u32_to_unit(b1.z), u32_to_unit(b1.w), u32_to_unit(b2.x)) - one;
    float3 p3 = 2.0f * f3(u32_to_unit(b2.y), u32_to_unit(b2.z), u32_to_unit(b2.w)) - one;
    bool a0 = mag_sq3(p0) < 1.0f, a1 = mag_sq3(p1) < 1.0f, a2 = mag_sq3(p2) < 1.0f, a3 = mag_sq3(p3) < 1.0f;
    if (a0 || a1 || a2 || a3) {
        int used = a0 ? 3 : (a1 ? 6 : (a2 ? 9 : 12));
        float3 p = a0 ? p0 : (a1 ? p1 : (a2 ? p2 : p3));
        // leave the stream where the sequential loop would have left it
        rng.idx = (uint32_t)used;
        rng.buf = used <= 3 ? b0 : (used <= 6 ? b1 : b2);
        return p;
    }
    rng.idx = 12u;
    return random_in_unit_sphere(rng);
}
FW_DEV float3 random_in_unit_sphere_fresh(ArrayStream& rng) { return random_in_unit_sphere(rng); }

// util.rs:45-52
template <class Stream>
FW_DEV float3 random_in_unit_disk(Stream& rng) {
    for (;;) {
        float a = rng.next(), b = rng.next();
        float3 p = 2.0f * f3(a, b, 0.0f) - f3(1.0f, 1.0f, 0.0f);
        if (dot3(p, p) < 1.0f) return p;
    }
}
FW_DEV float3 reflect3(float3 v, float3 n) { return v - 2.0f * dot3(v, n) * n; }  // util.rs:54-56
FW_DEV bool refract3(float3 v, float3 n, float ni_over_nt, float3& out) {        // util.rs:58-67
    float3 uv = normalized3(v);
    float dt = dot3(uv, n);
    float disc = 1.0f - ni_over_nt * ni_over_nt * (1.0f - dt * dt);
    if (disc > 0.0f) {
        out = ni_over_nt * (uv - n * dt) - n * sqrtf(disc);
        return true;
    }
    return false;
}
FW_DEV float schlick(float cosine, float ref_idx) {  // util.rs:69-73
    float r0 = (1.0f - ref_idx) / (1.0f + ref_idx);
    r0 = r0 * r0;
    return r0 + (1.0f - r0) * powf(1.0f - cosine, 5.0f);
}

struct ScatterOut {
    bool scattered;
    float3 attenuation, origin, dir;
};

// One material at a time — each is the body of its own shade kernel.
template <class Stream>
FW_DEV void scatter_lambertian(const DeviceScene& S, int tex, float3 point, float3 normal, float2 uv, Stream& rng,
                               ScatterOut& out) {
    float3 target = point + normal + random_in_unit_sphere_fresh(rng);
    out.origin = point;
    out.dir = target - point;
    out.attenuation = texture_sample(S, tex, uv, point);
    out.scattered = true;
}
template <class Stream>
FW_DEV void scatter_metal(float3 albedo, float roughness, float3 in_dir, float3 point, float3 normal, Stream& rng,
                          ScatterOut& out) {
    float3 reflected = reflect3(in_dir, normal);
    out.origin = point;
    out.dir = reflected + roughness * random_in_unit_sphere_fresh(rng);
    out.attenuation = albedo;
    out.scattered = dot3(out.dir, normal) > 0.0f;
}
template <class Stream>
FW_DEV void scatter_dielectric(float ref_idx, float3 in_dir, float3 point, float3 normal, Stream& rng, ScatterOut& out) {
    float3 reflected = reflect3(in_dir, normal);
    float3 outward_normal;
    float ni_over_nt, cosine;
    if (dot3(in_dir, normal) > 0.0f) {
        outward_normal = -normal;
        ni_over_nt = ref_idx;
        cosine = ref_idx * dot3(in_dir, normal) / mag3(in_dir);
    } else {
        outward_normal = normal;
        ni_over_nt = 1.0f / ref_idx;
        cosine = -dot3(in_dir, normal) / mag3(in_dir);
    }
    out.origin = point;
    out.attenuation = f3(1.0f, 1.0f, 1.0f);
    out.scattered = true;
    float3 refracted;
    if (refract3(in_dir, outward_normal, ni_over_nt, refracted)) {
        if (rng.next() > schlick(cosine, ref_idx)) {
            out.dir = refracted;
            return;
        }
    }
    out.dir = reflected;
}
template <class Stream>
FW_DEV void scatter_isotropic(const DeviceScene& S, int tex, float3 point, float2 uv, Stream& rng, ScatterOut& out) {
    out.attenuation = texture_sample(S, tex, uv, point);
    out.origin = point;
    out.dir = random_in_unit_sphere_fresh(rng);
    out.scattered = true;
}

}  // namespace fw
