// shade.cuh — scattering, texture lookup and miss radiance.
//   v2     MetalBSDF / DielectricBSDF / DiffuseBSDF      taichi_pathtracer/10_final/bsdf.py:5-110
//   legacy gen_secondary_rays + sample_* + cal_reflectivity_*   legacy/PT_in_one_weekend/15_module.py:281-347,994-1013
//   bilinear / environment_color                           15_module.py:238-258,970-977
// Same decisions and distributions as the reference; transcendental functions use the fast MUFU paths
// (the reference runs under Taichi's fast_math too), so agreement with the oracle is statistical.
#pragma once
#include "extend.cuh"

struct PathState {
    float3 o, d, l;
    uint32_t pixel, sample, bounce;
};

// ---- sampling helpers ----------------------------------------------------------------------
PT_DEV float3 sample_at_sphere(float u0, float u1) {  // bsdf.py:5-12, 15_module.py:295-302
    float z = 1.0f - 2.0f * u0;
    float r = sqrtf(fmaxf(0.0f, 1.0f - z * z));
    float s, c;
    sincos_2pi(u1, &s, &c);
    return f3(r * c, r * s, z);
}
PT_DEV float3 sample_lambertian(float3 n, float u0, float u1) {  // bsdf.py:15-18
    return normalize(n + sample_at_sphere(u0, u1));
}
PT_DEV float3 reflect_dir(float3 d, float3 n) {  // bsdf.py:40-44
    return d + (-2.0f * dot(d, n)) * n;
}
PT_DEV float3 slerp_dir(float3 a, float3 b, float t) {  // bsdf.py:21-27
    if (t == 0.0f) return normalize(a);  // sin(omega)/sin(omega) = 1, sin(0) = 0: exactly a
    float dd = fminf(fmaxf(dot(a, b), -1.0f), 1.0f);
    float omega = acosf(dd);
    float so = __sinf(omega);
    float3 o;
    if (so < 1e-6f) {
        o = (1.0f - t) * a + t * b;
    } else {
        float inv = 1.0f / so;
        o = (__sinf((1.0f - t) * omega) * inv) * a + (__sinf(t * omega) * inv) * b;
    }
    return normalize(o);
}
PT_DEV float3 sample_micro_normal(float3 d, float3 n, float roughness, float u0, float u1) {  // bsdf.py:30-37
    float3 s = sample_lambertian(n, u0, u1);
    float3 r = reflect_dir(d, n);
    r = slerp_dir(r, s, roughness * roughness);
    return normalize(r - d);
}
PT_DEV float3 refract_dir(float3 d, float3 n, float ior) {  // bsdf.py:47-59
    float k = dot(d, n);
    float3 perp = (d - k * n) * (1.0f / ior);
    float len2 = dot(perp, perp);
    if (len2 > 1.0f) return reflect_dir(d, n);
    return perp - sqrtf(1.0f - len2) * n;
}

// ---- surface attributes at a hit ----------------------------------------------------------------
// The scatter code and the denoiser's first-hit features (denoise.cu) read a surface through these, so both see the
// same normal and albedo.  Outward normals: the caller turns them to face the ray.
PT_DEV float3 sphere_normal_v2(float4 cr, float3 point) {  // world.py:58
    return normalize(point - f3(cr));
}

// ---- v2 scatter: one propagate_once hit branch (__main__.py:65-75) -----------------------------
// mat0 = albedo.rgb, roughness ; mat1 = bits(metallic), ior, bits(transparency), _
PT_DEV void scatter_v2(const SceneView& sv, PathState& p, const Hit& h, int shading_model, uint32_t seed) {
    const float4 cr = __ldg(&sv.sph_cr[h.prim]);
    const float4 m0 = __ldg(&sv.sph_mat[2 * h.prim]);
    const float4 m1 = __ldg(&sv.sph_mat[2 * h.prim + 1]);
    const float3 albedo = f3(m0);
    const float3 point = p.o + h.t * p.d;            // world.py:57
    float3 normal = sphere_normal_v2(cr, point);
    float ior = m1.y;
    if (dot(p.d, normal) > 0.0f) {                   // world.py:31-33
        normal = -normal;
        ior = 1.0f / ior;
    }
    const float4 u = rng4(p.pixel, p.sample, 1u + 2u * p.bounce, seed);
    p.o = point;
    if (shading_model == PT_SHADE_V2_DIFFUSE) {      // 6_diffuse/bsdf.py:20-26
        p.l = p.l * albedo;
        p.d = sample_lambertian(normal, u.x, u.y);
        return;
    }
    const float3 d = p.d;
    const float3 n = sample_micro_normal(d, normal, m0.w, u.x, u.y);
    const float cos_theta = fmaxf(0.0f, -dot(n, d));
    const float w = pow5(1.0f - cos_theta);
    if (__float_as_int(m1.x) == 1) {                 // MetalBSDF bsdf.py:71-86
        p.l = p.l * f3(albedo.x + (1.0f - albedo.x) * w, albedo.y + (1.0f - albedo.y) * w,
                       albedo.z + (1.0f - albedo.z) * w);
        p.d = reflect_dir(d, n);
    } else {                                         // DielectricBSDF bsdf.py:89-110
        float f0 = (ior - 1.0f) / (ior + 1.0f);
        f0 *= f0;
        const float F = f0 + (1.0f - f0) * w;
        if (u.z > F) {
            p.l = p.l * albedo;
            if (__float_as_int(m1.z) != 0) {
                p.d = refract_dir(d, n, ior);
            } else {
                const float4 u2 = rng4(p.pixel, p.sample, 2u + 2u * p.bounce, seed);
                p.d = sample_lambertian(normal, u2.x, u2.y);
            }
        } else {
            p.d = reflect_dir(d, n);
        }
    }
}

// stages 4-5 (5_anti_aliasing/__main__.py:19-28): the outward geometric normal as a colour, path ends at the hit
PT_DEV float3 normal_color(const SceneView& sv, const PathState& p, const Hit& h) {
    const float4 cr = __ldg(&sv.sph_cr[h.prim]);
    const float3 n = normalize(p.o + h.t * p.d - f3(cr));
    return f3(0.5f * (n.x + 1.0f), 0.5f * (n.y + 1.0f), 0.5f * (n.z + 1.0f));
}

PT_DEV float3 sky_color(float3 d) {  // backbround_color, __main__.py:58-62
    float t = 0.5f * (d.y + 1.0f);
    return f3((1.0f - t) + t * 0.5f, (1.0f - t) + t * 0.7f, (1.0f - t) + t);
}

// ---- legacy textures ------------------------------------------------------------------------
// ti.mod (Python modulo) by the area width w > 0, without an integer division: floor(a / w) from the float
// reciprocal is off by at most one for |a| < 2^23 (texture coordinates that tile many times still are), and the
// remainder is corrected by one step.  Tiling uvs (ground plane) made the generic a % m a hot spot.
PT_DEV int pymod_w(int a, int w, float inv_w) {
    const int q = __float2int_rd((float)a * inv_w);
    int r = a - q * w;
    if (r < 0) r += w;
    else if (r >= w) r -= w;
    return r;
}

struct Taps {
    int l, r, b, t;
    float lb, lt, rb, rt;
};
// bilinear (15_module.py:238-258), quirks kept: truncating cast after -0.5; v wraps with the area WIDTH
PT_DEV Taps bilinear_taps(int4 area, float u, float v) {
    const int w = area.z - area.x, hgt = area.w - area.y;
    Taps k;
    u = u * (float)w - 0.5f;
    v = v * (float)hgt - 0.5f;
    const int l = (int)u, r = l + 1, b = (int)v, t = b + 1;
    k.lb = ((float)r - u) * ((float)t - v);
    k.lt = ((float)r - u) * (v - (float)b);
    k.rb = (u - (float)l) * ((float)t - v);
    k.rt = (u - (float)l) * (v - (float)b);
    const float inv_w = 1.0f / (float)w;
    const int ml = pymod_w(l, w, inv_w), mb = pymod_w(b, w, inv_w);  // (x + 1) mod w follows from x mod w
    k.l = area.x + ml;
    k.r = area.x + (ml + 1 >= w ? ml + 1 - w : ml + 1);
    k.b = area.y + mb;
    k.t = area.y + (mb + 1 >= w ? mb + 1 - w : mb + 1);
    return k;
}

struct Texel {
    float3 albedo, normal;
    float roughness, metallic;
};
// `lut` = the three 256-entry transfer tables (albedo^2.2 | x^2 | 2x-1).  The persistent render kernel hands in its
// SHARED-memory copy (3 KB per block, filled once per launch): round 1's ncu listing showed ~25 scalar global loads per
// textured hit for them; the other kernel forms pass sv.lut (global).
PT_DEV void texel_accum(const SceneView& sv, const float* lut, int x, int y, float wgt, bool want_normal, Texel& o) {
    if (x < 0 || y < 0 || x >= sv.tex_W || y >= sv.tex_H) return;  // outside the field: zero
    const uint2 q = __ldcg(&sv.atlas[(size_t)x * sv.tex_H + y]);  // L2 only: the atlas must not evict BVH nodes from L1
    const float* la = lut;
    const float* ls = lut + 256;
    o.albedo.x = fmaf(wgt, la[q.x & 255u], o.albedo.x);
    o.albedo.y = fmaf(wgt, la[(q.x >> 8) & 255u], o.albedo.y);
    o.albedo.z = fmaf(wgt, la[(q.x >> 16) & 255u], o.albedo.z);
    o.roughness = fmaf(wgt, ls[q.x >> 24], o.roughness);
    o.metallic = fmaf(wgt, ls[q.y >> 24], o.metallic);
    if (want_normal) {
        const float* ln = lut + 512;
        o.normal.x = fmaf(wgt, ln[q.y & 255u], o.normal.x);
        o.normal.y = fmaf(wgt, ln[(q.y >> 8) & 255u], o.normal.y);
        o.normal.z = fmaf(wgt, ln[(q.y >> 16) & 255u], o.normal.z);
    }
}
// The four taps of a bilinear lookup, straight-line: a tap outside the field reads a clamped address and gets weight 0
// ("reads outside the field are 0", as the reference's out-of-range field access) instead of branching around its load.
// With one early-return branch per tap (round 1) the compiler could not move a load across the reconvergence point, so
// the four L2 loads of a lookup ran one after the other; now all four are in flight together.  Same taps, same order
// of accumulation, fma(0, x, o) = o: the result is bit-identical.
PT_DEV Texel sample_texture(const SceneView& sv, const float* lut, int id, float u, float v, bool want_normal) {
    Texel o;
    o.albedo = f3(0, 0, 0); o.normal = f3(0, 0, 0); o.roughness = 0.0f; o.metallic = 0.0f;
    if (id < 0 || id >= sv.ntex) return o;
    if (__ldg(&sv.tex_flags[id]) & 1) {  // plain diffuse map: constant normal (0,0,1), 15_module.py:84,104
        want_normal = false;
        o.normal = f3(0.0f, 0.0f, 1.0f);
    }
    const Taps k = bilinear_taps(__ldg(&sv.tex_areas[id]), u, v);
#ifdef PT_OPT_BRANCHY_TAPS
    texel_accum(sv, lut, k.l, k.b, k.lb, want_normal, o);
    texel_accum(sv, lut, k.l, k.t, k.lt, want_normal, o);
    texel_accum(sv, lut, k.r, k.b, k.rb, want_normal, o);
    texel_accum(sv, lut, k.r, k.t, k.rt, want_normal, o);
#else
    const bool in_l = (unsigned)k.l < (unsigned)sv.tex_W, in_r = (unsigned)k.r < (unsigned)sv.tex_W;
    const bool in_b = (unsigned)k.b < (unsigned)sv.tex_H, in_t = (unsigned)k.t < (unsigned)sv.tex_H;
    const size_t row_l = (size_t)(in_l ? k.l : 0) * sv.tex_H, row_r = (size_t)(in_r ? k.r : 0) * sv.tex_H;
    const int yb = in_b ? k.b : 0, yt = in_t ? k.t : 0;
    const uint2 q0 = __ldcg(&sv.atlas[row_l + yb]), q1 = __ldcg(&sv.atlas[row_l + yt]);   // L2 only: the atlas must not
    const uint2 q2 = __ldcg(&sv.atlas[row_r + yb]), q3 = __ldcg(&sv.atlas[row_r + yt]);   // evict BVH nodes from L1
    const float w0 = in_l && in_b ? k.lb : 0.0f, w1 = in_l && in_t ? k.lt : 0.0f;
    const float w2 = in_r && in_b ? k.rb : 0.0f, w3 = in_r && in_t ? k.rt : 0.0f;
    const float* la = lut;
    const float* ls = lut + 256;
    const uint2 q[4] = {q0, q1, q2, q3};
    const float w[4] = {w0, w1, w2, w3};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        o.albedo.x = fmaf(w[i], la[q[i].x & 255u], o.albedo.x);
        o.albedo.y = fmaf(w[i], la[(q[i].x >> 8) & 255u], o.albedo.y);
        o.albedo.z = fmaf(w[i], la[(q[i].x >> 16) & 255u], o.albedo.z);
        o.roughness = fmaf(w[i], ls[q[i].x >> 24], o.roughness);
        o.metallic = fmaf(w[i], ls[q[i].y >> 24], o.metallic);
    }
    if (want_normal) {
        const float* ln = lut + 512;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            o.normal.x = fmaf(w[i], ln[q[i].y & 255u], o.normal.x);
            o.normal.y = fmaf(w[i], ln[(q[i].y >> 8) & 255u], o.normal.y);
            o.normal.z = fmaf(w[i], ln[(q[i].y >> 16) & 255u], o.normal.z);
        }
    }
#endif
    return o;
}
PT_DEV float3 env_fetch(const SceneView& sv, int x, int y) {
    if (x < 0 || y < 0 || x >= sv.env_W || y >= sv.env_H) return f3(0, 0, 0);
    return f3(__ldcg(&sv.env[(size_t)x * sv.env_H + y]));
}
PT_DEV float3 environment_color(const SceneView& sv, float3 d) {  // 15_module.py:970-977
    if (!sv.has_env) return sky_color(d);
#ifdef PT_OPT_LIBM_TRIG
    const float phi = asinf(fminf(fmaxf(d.y, -1.0f), 1.0f));
    const float theta = atan2f(-d.x, -d.z);
#else
    const float phi = fast_asinf(d.y);
    const float theta = fast_atan2f(-d.x, -d.z);
#endif
    const float u = (theta * (1.0f / PT_PI) + 1.0f) * 0.5f;
    const float v = phi * (1.0f / PT_PI) + 0.5f;
    const Taps k = bilinear_taps(sv.env_area, u, v);
#ifdef PT_OPT_BRANCHY_TAPS
    return k.lb * env_fetch(sv, k.l, k.b) + k.lt * env_fetch(sv, k.l, k.t) + k.rb * env_fetch(sv, k.r, k.b) +
           k.rt * env_fetch(sv, k.r, k.t);
#else
    const bool in_l = (unsigned)k.l < (unsigned)sv.env_W, in_r = (unsigned)k.r < (unsigned)sv.env_W;
    const bool in_b = (unsigned)k.b < (unsigned)sv.env_H, in_t = (unsigned)k.t < (unsigned)sv.env_H;
    const size_t row_l = (size_t)(in_l ? k.l : 0) * sv.env_H, row_r = (size_t)(in_r ? k.r : 0) * sv.env_H;
    const int yb = in_b ? k.b : 0, yt = in_t ? k.t : 0;
    const float4 e0 = __ldcg(&sv.env[row_l + yb]), e1 = __ldcg(&sv.env[row_l + yt]);
    const float4 e2 = __ldcg(&sv.env[row_r + yb]), e3 = __ldcg(&sv.env[row_r + yt]);
    const float3 z = f3(0, 0, 0);   // selects, not weights: an HDR texel may be anything, 0 * inf would not be 0
    return k.lb * (in_l && in_b ? f3(e0) : z) + k.lt * (in_l && in_t ? f3(e1) : z) + k.rb * (in_r && in_b ? f3(e2) : z) +
           k.rt * (in_r && in_t ? f3(e3) : z);
#endif
}

// ---- legacy scatter ----------------------------------------------------------------------------
PT_DEV float3 sample_in_sphere(float u0, float u1, float u2) {  // 15_module.py:304-312
    const float r = cbrtf(u0);
    float st, ct;
    sincos_2pi(u1, &st, &ct);
    const float cphi = u2 * 2.0f - 1.0f;  // cos(acos(x)) = x, sin(acos(x)) = sqrt(1 - x^2)
    const float sphi = sqrtf(fmaxf(0.0f, 1.0f - cphi * cphi));
    return f3(r * ct * sphi, r * st * sphi, r * cphi);
}

struct LegacySurface {
    float3 normal, albedo;  // outward shading normal (normal-mapped on spheres), texture albedo
    float roughness, metallic;
    int transparency;
};
PT_DEV LegacySurface legacy_surface(const SceneView& sv, const float* lut, const Hit& h, float3 point) {
    LegacySurface o;
    o.transparency = 0;
    if (h.prim < sv.n_sph) {  // sphere_hit, 15_module.py:864-896
        const float4 cr = __ldg(&sv.sph_cr[h.prim]);
        const float4 aux = __ldg(&sv.sph_aux[h.prim]);
        const float3 N = normalize(point - f3(cr));
        const float r = sqrtf(N.x * N.x + N.z * N.z);
        const float3 T = f3(N.z / r, 0.0f, -N.x / r);
        const float3 B = f3(N.x * N.y, -r, N.z * N.y);
        const float phi = asinf(fminf(fmaxf(N.y, -1.0f), 1.0f));
        const float theta = atan2f(-N.x, -N.z);
        const float uu = (theta * (1.0f / PT_PI) + 1.0f) * 0.5f;
        const float vv = phi * (1.0f / PT_PI) + 0.5f;
        const Texel tx = sample_texture(sv, lut, __float_as_int(aux.z), 2.0f * uu, vv, true);
        o.normal = normalize(tx.normal.x * T + tx.normal.y * B + tx.normal.z * N);
        o.albedo = tx.albedo; o.roughness = tx.roughness; o.metallic = tx.metallic;
        o.transparency = __float_as_int(aux.y);
    } else {  // triangle_hit, 15_module.py:929-950
        const float4* s = sv.tri_shade + 4 * (size_t)(h.prim - sv.n_sph);
        const float4 s0 = __ldcg(s), s1 = __ldcg(s + 1), s2 = __ldcg(s + 2), s3 = __ldcg(s + 3);
        const float w1 = 1.0f - h.u - h.v, w2 = h.u, w3 = h.v;
        o.normal = normalize(w1 * f3(s0) + w2 * f3(s1) + w3 * f3(s2));
        const float uu = w1 * s0.w + w2 * s2.w + w3 * s3.y;
        const float vv = w1 * s1.w + w2 * s3.x + w3 * s3.z;
        const Texel tx = sample_texture(sv, lut, __float_as_int(s3.w), uu, vv, false);
        o.albedo = tx.albedo; o.roughness = tx.roughness; o.metallic = tx.metallic;
    }
    return o;
}

// propagate_once hit branch (15_module.py:983-989) + gen_secondary_rays (:994-1013)
PT_DEV void scatter_legacy(const SceneView& sv, PathState& p, const Hit& h, float absorptivity, uint32_t seed,
                           const float* lut) {
    const float3 d = p.d;
    const float3 point = p.o + h.t * d;
    const LegacySurface sf = legacy_surface(sv, lut, h, point);
    float3 normal = sf.normal;
    const float3 albedo = sf.albedo;
    const float roughness = sf.roughness, metallic = sf.metallic;
    const int transparency = sf.transparency;
    float ior = 1.5f;
    if (dot(d, normal) > 0.0f) {  // 15_module.py:985-988
        normal = -normal;
        ior = 1.0f / ior;
        absorptivity = 0.0f;
    }
    const float4 u = rng4(p.pixel, p.sample, 1u + 2u * p.bounce, seed);
    const float ndd = 1.0f + dot(normal, d);
    const float w = pow5(ndd);
    bool mirror;  // sample_reflect branch
    if (u.x < metallic) {  // :997-1000, cal_reflectivity_metal :281-285
        p.l = p.l * f3(albedo.x + (1.0f - albedo.x) * w, albedo.y + (1.0f - albedo.y) * w,
                       albedo.z + (1.0f - albedo.z) * w);
        mirror = true;
    } else {
        float f0 = (ior - 1.0f) / (ior + 1.0f);
        f0 *= f0;
        const float F = f0 + (1.0f - f0) * w;  // cal_reflectivity_dielectirc :288-292
        mirror = !(u.y > F);
        if (!mirror) {
            p.l = p.l * (albedo * (1.0f - absorptivity));
            if (transparency) {  // sample_refract :337-347 (clamps, no TIR branch)
                const float4 u2 = rng4(p.pixel, p.sample, 2u + 2u * p.bounce, seed);
                const float3 s = sample_in_sphere(u.z, u.w, u2.x);
                const float k = dot(d, normal);
                const float3 perp = (d - k * normal) * (1.0f / ior);
                const float len2 = fminf(dot(perp, perp), 1.0f);
                p.d = normalize(perp - sqrtf(1.0f - len2) * normal + roughness * s);
            } else {  // sample_diffuse :322-325
                p.d = normalize(normal + sample_at_sphere(u.z, u.w));
            }
        }
    }
    if (mirror) {  // sample_reflect :329-334
        const float4 u2 = rng4(p.pixel, p.sample, 2u + 2u * p.bounce, seed);
        const float3 s = sample_in_sphere(u.z, u.w, u2.x);
        p.d = normalize(reflect_dir(d, normal) + roughness * s);
    }
    p.o = point + (2.0f * PT_EPS) * normal;  // :1013
}

// ---- legacy tutorial stages 6 / 7 (untextured) ---------------------------------------------------
// legacy/PT_in_one_weekend/7_reflect.py:187-209 (propagate_once) with :49-96 (cal_reflectivity_*, sample_*) and
// 6_diffuse.py:160-170.  These are the functions 15_module.py:281-334 still uses, on constant-material spheres under
// the sky gradient — the only form of the legacy scattering model whose converged renders are in the reference
// checkout (legacy/PT_in_one_weekend/{6_diffuse,7_reflect}.png).  No back-face flip (a sphere is only ever met from
// outside: World.hit keeps the near root and t > 1e-3), no origin offset.
PT_DEV void scatter_legacy_stage(const SceneView& sv, PathState& p, const Hit& h, int shading_model, float absorptivity,
                                 uint32_t seed) {
    const float4 cr = __ldg(&sv.sph_cr[h.prim]);
    const float4 m0 = __ldg(&sv.sph_mat[2 * h.prim]);
    const float4 m1 = __ldg(&sv.sph_mat[2 * h.prim + 1]);
    const float3 albedo = f3(m0), d = p.d;
    const float3 point = p.o + h.t * d;
    const float3 normal = normalize(point - f3(cr));
    const float4 u = rng4(p.pixel, p.sample, 1u + 2u * p.bounce, seed);
    p.o = point;
    if (shading_model == PT_SHADE_LEGACY_STAGE6) {  // 6_diffuse.py:165-167
        p.l = absorptivity * p.l * albedo;
        p.d = normalize(normal + sample_at_sphere(u.z, u.w));
        return;
    }
    const float w = pow5(1.0f + dot(normal, d));
    bool mirror;
    if (__float_as_int(m1.x) != 0) {  // metallic: cal_reflectivity_metal, 7_reflect.py:49-53,191-194
        p.l = p.l * f3(albedo.x + (1.0f - albedo.x) * w, albedo.y + (1.0f - albedo.y) * w, albedo.z + (1.0f - albedo.z) * w);
        mirror = true;
    } else {  // cal_reflectivity_dielectirc :56-60, the coin :197
        float f0 = (m1.y - 1.0f) / (m1.y + 1.0f);
        f0 *= f0;
        mirror = !(u.y > f0 + (1.0f - f0) * w);
        if (!mirror) {  // :198-199
            p.l = p.l * (albedo * absorptivity);
            p.d = normalize(normal + sample_at_sphere(u.z, u.w));
        }
    }
    if (mirror) {  // sample_reflect :91-96: the lobe shrinks with k = -d.n (15_module.py:329-334 dropped that factor)
        const float4 u2 = rng4(p.pixel, p.sample, 2u + 2u * p.bounce, seed);
        const float3 s = sample_in_sphere(u.z, u.w, u2.x);
        const float k = -dot(d, normal);
        p.d = normalize(d + (2.0f * k) * normal + (k * m0.w) * s);
    }
}

// ---- camera: Camera.get_rays (camera.py:71-93, 15_module.py:438-453) ---------------------------
struct CameraDev {
    float3 pos, front, right, up;
    float view_w, view_h, focal, aperture;
    float inv_w, inv_h;  // 1/width, 1/height (PT_FLAG_PIXEL_GRID: 1/(width-1), 1/(height-1))
    float jitter;        // 1 (pixel jitter, camera.py:88) or 0 (PT_FLAG_PIXEL_GRID); x * 1.0f is exact
};
PT_DEV void camera_ray(const CameraDev& c, int i, int j, float4 u, float3* o, float3* d) {
    const float fx = ((float)i + u.x * c.jitter) * c.inv_w - 0.5f;
    const float fy = ((float)j + u.y * c.jitter) * c.inv_h - 0.5f;
    const float3 target = c.focal * (c.front + (fx * c.view_w) * c.right + (fy * c.view_h) * c.up);
    if (c.aperture == 0.0f) {  // pinhole (warp-uniform): the lens sample is multiplied by zero in the reference, skip it
        *o = c.pos;
        *d = normalize(target);
        return;
    }
    const float r = sqrtf(u.z);  // sample_in_disk, camera.py:29-35
    float s, cs;
    sincos_2pi(u.w, &s, &cs);
    const float3 origin = (0.5f * c.aperture) * ((r * cs) * c.right + (r * s) * c.up);
    *o = c.pos + origin;
    *d = normalize(target - origin);
}
