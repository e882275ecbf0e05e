// fp32 shading: Material::evaluate (material.rs:91-109, pdf=None as radiance() passes it,
// lib.rs:532) and Scene::background (lib.rs:254-285).
//
// The reference evaluates brdf * cos / pdf literally; the microfacet density D appears in
// both the BRDF and the sampling pdf and cancels (exactly for CookTorrance::scatter, where
// Pdf::value and Brdf::brdf rebuild the same half vector, material.rs:917,927 vs 1287,1298;
// to rounding for the glass variants).  The kernels evaluate the cancelled closed forms:
//     reflection  : color * F * G * (h.l) / (n.v)            (material.rs:721-758,1276-1322)
//     refraction  : color * (1-F) * G * (h.v) / (n.v)        (material.rs:764-812,1362-1442)
// with G = min(2 nh nv / hv, 2 nh nl / hv, 1) (Cook-Torrance V-cavity term) and Schlick F.
// This keeps the reference's *estimator* (including the missing cos(theta_h) factor in the
// half-vector pdf, SURVEY.md F2) and all of its NoScatter conditions.
#pragma once
#include "device_types.cuh"

namespace rrs {

#define RRS_PI_F 3.14159265358979323846f

struct ScatterOut {
    bool scatter;
    float3 color;
    float3 dir;
};

__device__ __forceinline__ float powi5f(float a) {
    float a2 = a * a;
    return a * (a2 * a2);
}

// Vec3::orthonormal_basis vecmath.rs:341-352
__device__ __forceinline__ void orthonormal_basis(float3 n, float3& e1, float3& e2) {
    if (fabsf(n.x) > fabsf(n.y))
        e1 = normalize3(f3(n.z, 0.f, -n.x));
    else
        e1 = normalize3(f3(0.f, n.z, -n.y));
    e2 = normalize3(cross3(n, e1));
}

// material.rs:1472-1479
__device__ __forceinline__ float schlick_scalar(float r0, float cosv) { return r0 + (1.f - r0) * powi5f(1.f - cosv); }
// material.rs:1492-1496
__device__ __forceinline__ float3 reflect3(float3 n, float3 v) { return sub3(scale3(n, 2.f * dot3(v, n)), v); }
// material.rs:1502-1518
__device__ __forceinline__ bool refract3(float3 n, float3 v, float eta, float3& out) {
    float cos_t = dot3(v, n);
    float sin_t = sqrtf(fmaxf(0.f, 1.f - cos_t * cos_t));
    if (eta * sin_t > 1.f) return false;
    float3 par = scale3(sub3(scale3(n, cos_t), v), eta);
    float perp = -sqrtf(fmaxf(0.f, 1.f - dot3(par, par)));
    out = madd3(n, perp, par);
    return true;
}

// Pdf::Cosine generate material.rs:982-993
__device__ __forceinline__ float3 cosine_sample(float3 n, float u, float uphi) {
    float3 e1, e2;
    orthonormal_basis(n, e1, e2);
    float s, c;
    sincospif(2.f * uphi, &s, &c);
    float su = sqrtf(u);
    float x = c * su, y = s * su, z = sqrtf(1.f - u);
    return add3(add3(scale3(e1, x), scale3(e2, y)), scale3(n, z));
}

// Beckmann half-vector about n: material.rs:1006-1020 / 1137-1161
__device__ __forceinline__ float3 beckmann_sample(float alpha2, float3 n, float uphi, float uxi) {
    float3 e1, e2;
    orthonormal_basis(n, e1, e2);
    float s, c;
    sincospif(2.f * uphi, &s, &c);
    float tan2 = -alpha2 * logf(1.f - uxi);
    float cost = rsqrtf(1.f + tan2);
    float sint = sqrtf(fmaxf(0.f, 1.f - cost * cost));
    return add3(add3(scale3(e1, c * sint), scale3(e2, s * sint)), scale3(n, cost));
}

__device__ __forceinline__ float3 fresnel_ct(const DMat& m, bool metallic, float hv) {
    if (metallic) {
        float w = powi5f(1.f - hv);
        float3 r0 = xyz(m.m1);
        return f3(r0.x + (1.f - r0.x) * w, r0.y + (1.f - r0.y) * w, r0.z + (1.f - r0.z) * w);
    }
    float f = schlick_scalar(m.m2.z, hv);
    return f3(f, f, f);
}

// CookTorrance::evaluate_reflection (material.rs:721-758) with brdf (1276-1322) and the
// Beckmann pdf cancelled.  n, h are in the hemisphere the caller chose; `div` is an extra
// divisor (Fresnel importance sampling in Plastic / CookTorranceGlass), 1 otherwise.
// fresnel_mode: 0 = Schlick metallic r0 (m1), 1 = Schlick dielectric, 2 = none (the caller's
// division by the same Fresnel value cancels it: CookTorranceGlass reflect branch).
__device__ __forceinline__ ScatterOut ct_reflection(const DMat& m, float3 color, int fresnel_mode, float3 n, float3 h,
                                                    float3 v, float3 l, float div) {
    ScatterOut r;
    r.scatter = false;
    r.color = f3(0, 0, 0);
    r.dir = l;
    if (dot3(h, v) < 0.f) return r;
    float nl_s = dot3(n, l);
    if (nl_s < 0.f) return r;
    float nv = fabsf(dot3(n, v));
    float nl = fabsf(nl_s);
    float3 hh = add3(v, l);
    if (nv == 0.f || nl == 0.f) return r;
    if (hh.x == 0.f && hh.y == 0.f && hh.z == 0.f) return r;
    hh = normalize3(hh);
    float nh = dot3(n, hh);
    float hv = dot3(hh, v);
    float g = fminf(2.f * nh * nv / hv, fminf(2.f * nh * nl / hv, 1.f));
    float w = g * dot3(h, l) / nv;
    float3 c;
    if (fresnel_mode == 2) {
        c = scale3(color, w);
    } else {
        float3 F = fresnel_ct(m, fresnel_mode == 0, hv);
        c = scale3(mul3(color, F), w / div);
    }
    if (c.x == 0.f && c.y == 0.f && c.z == 0.f) return r;
    r.scatter = true;
    r.color = c;
    return r;
}

// CookTorrance::evaluate_refraction (material.rs:764-812) with btdf (1362-1442) cancelled.
// keep_one_minus_f: CookTorranceRefract keeps the (1-F) factor; CookTorranceGlass divides it out.
__device__ __forceinline__ ScatterOut ct_refraction(const DMat& m, float3 color, float3 n, float3 h, float3 v, float3 l,
                                                    bool keep_one_minus_f) {
    ScatterOut r;
    r.scatter = false;
    r.color = f3(0, 0, 0);
    r.dir = l;
    if (dot3(h, v) < 0.f) return r;
    float nl_s = dot3(n, l);
    if (nl_s > 0.f) return r;
    float nv = fabsf(dot3(n, v));
    float nl = fabsf(nl_s);
    if (nv == 0.f || nl == 0.f) return r;
    float hv = fabsf(dot3(h, v));
    float nh = dot3(n, h);
    float g = fminf(2.f * nh * nv / hv, fminf(2.f * nh * nl / hv, 1.f));
    float w = g * hv / nv;
    if (keep_one_minus_f) w *= 1.f - schlick_scalar(m.m2.z, dot3(h, v));
    float3 c = scale3(color, w);
    if (c.x == 0.f && c.y == 0.f && c.z == 0.f) return r;
    r.scatter = true;
    r.color = c;
    return r;
}

// Material::evaluate, one inlined arm per variant (the reference's own shape, material.rs:91-109).  Fastest when
// a warp holds one material family — the sphere-series path loop uses it (gpurun_out/sweep_mat.log: +5 % there);
// material_evaluate_staged below is the form for mixed warps.  tests/test_gpu_render.py renders every material
// through both and compares.
__device__ __forceinline__ ScatterOut material_evaluate_cases(const DMat& m, float3 n, float3 v, float u0, float u1, float u2) {
    ScatterOut r;
    r.scatter = false;
    r.color = f3(0, 0, 0);
    r.dir = f3(0, 0, 0);
    const uint32_t tag = __float_as_uint(m.m0.w);
    const float3 color = xyz(m.m0);
    const float alpha2 = m.m1.w;
    const float ior = m.m2.x;
    switch (tag) {
        case RRS_MAT_LAMBERTIAN: {  // material.rs:259-281: (color/pi * n.l) / (n.l/pi) == color
            r.dir = cosine_sample(n, u0, u1);
            r.color = color;
            r.scatter = true;
            return r;
        }
        case RRS_MAT_REFLECT: {  // material.rs:283-303: color / |n.l| * (n.l)
            float3 l = reflect3(n, v);
            float nl = dot3(n, l);
            r.dir = l;
            r.color = scale3(color, nl / fabsf(nl));
            r.scatter = true;
            return r;
        }
        case RRS_MAT_REFRACT: {  // material.rs:305-337
            bool entering = dot3(n, v) > 0.f;
            float3 nn = entering ? n : neg3(n);
            float3 l;
            if (!refract3(nn, v, entering ? 1.f / ior : ior, l)) return r;
            r.dir = l;
            r.color = dot3(l, v) > 0.f ? f3(0, 0, 0) : color;
            r.scatter = true;
            return r;
        }
        case RRS_MAT_GLASS: {  // material.rs:339-401
            float cos_t = dot3(n, v);
            bool entering = cos_t > 0.f;
            float3 nn = entering ? n : neg3(n);
            float sin2 = 1.f - cos_t * cos_t;
            float eta = entering ? 1.f / ior : ior;
            bool do_reflect = eta * eta * sin2 >= 1.f;
            if (!do_reflect) do_reflect = u0 < schlick_scalar(m.m2.z, dot3(nn, v));
            if (do_reflect) {
                float3 l = reflect3(nn, v);
                float nl = dot3(nn, l);
                r.dir = l;
                r.color = scale3(color, nl / fabsf(nl));
                r.scatter = true;
                return r;
            }
            float3 l;
            if (!refract3(nn, v, eta, l)) return r;
            r.dir = l;
            r.color = dot3(l, v) > 0.f ? f3(0, 0, 0) : color;
            r.scatter = true;
            return r;
        }
        case RRS_MAT_COOK_TORRANCE: {  // material.rs:403-424
            float3 h = beckmann_sample(alpha2, n, u0, u1);
            float3 l = reflect3(h, v);
            bool metallic = __float_as_uint(m.m2.y) == RRS_FRESNEL_METALLIC;
            return ct_reflection(m, color, metallic ? 0 : 1, n, h, v, l, 1.f);
        }
        case RRS_MAT_COOK_TORRANCE_REFRACT: {  // material.rs:426-467
            bool entering = dot3(n, v) > 0.f;
            float3 nn = entering ? n : neg3(n);
            float eta = entering ? 1.f / ior : ior;
            float3 h = beckmann_sample(alpha2, nn, u0, u1);
            if (!entering) h = neg3(h);
            float3 l;
            if (!refract3(h, v, eta, l)) return r;
            return ct_refraction(m, color, nn, h, v, l, true);
        }
        case RRS_MAT_COOK_TORRANCE_GLASS: {  // material.rs:469-565
            float3 h = beckmann_sample(alpha2, n, u0, u1);  // about the UNflipped normal
            bool entering = dot3(n, v) > 0.f;
            if (!entering) h = neg3(h);
            float3 nn = entering ? n : neg3(n);
            float cos_t = dot3(h, v);
            float eta = entering ? 1.f / ior : ior;
            float sin2 = 1.f - cos_t * cos_t;
            if (eta * eta * sin2 >= 1.f)  // total internal reflection: Fresnel kept, no division
                return ct_reflection(m, color, 1, nn, h, v, reflect3(h, v), 1.f);
            float fres = schlick_scalar(m.m2.z, cos_t);
            if (u2 < fres)  // F / F cancels
                return ct_reflection(m, color, 2, nn, h, v, reflect3(h, v), 1.f);
            float3 l;
            if (!refract3(h, v, eta, l)) return r;
            return ct_refraction(m, color, nn, h, v, l, false);
        }
        case RRS_MAT_PLASTIC: {  // material.rs:567-593
            float fres = schlick_scalar(m.m2.z, dot3(n, v));
            if (u0 < fres) {
                float3 h = beckmann_sample(alpha2, n, u1, u2);
                float3 l = reflect3(h, v);
                return ct_reflection(m, xyz(m.m1), 1, n, h, v, l, fres);
            }
            r.dir = cosine_sample(n, u1, u2);
            r.color = color;
            r.scatter = true;
            return r;
        }
        default:  // NoReflect material.rs:107
            return r;
    }
}

// Material::evaluate.  u0..u2: the bounce's uniforms, consumed in the reference's call order.
//
// The nine variants share most of their arithmetic — a direction sampled about an axis (cosine lobe or
// Beckmann half vector), a mirror reflection or a refraction about some vector, and one of two Cook-Torrance
// weight formulas — so the function is written as those four shared stages with a small per-variant
// selection in between, instead of one inlined copy of every stage per `case`: lanes of a warp that hold
// different materials run the shared stages together, and the shading code is a third of its former size
// (the fused kernel stalled on instruction fetch, profiles/r01h_c3_frosted_*).  Each variant still performs
// exactly the operations of its reference arm:
//   LambertianDiffuse material.rs:259-281   Reflect :283-303   Refract :305-337   Glass :339-401
//   CookTorrance :403-424   CookTorranceRefract :426-467   CookTorranceGlass :469-565   Plastic :567-593
__device__ __forceinline__ ScatterOut material_evaluate_staged(const DMat& m, float3 n, float3 v, float u0, float u1, float u2) {
    ScatterOut r;
    r.scatter = false;
    r.color = f3(0, 0, 0);
    r.dir = f3(0, 0, 0);
    const uint32_t tag = __float_as_uint(m.m0.w);
    const float3 color = xyz(m.m0);
    const float alpha2 = m.m1.w;
    const float ior = m.m2.x;
    const float nv_s = dot3(n, v);
    const bool entering = nv_s > 0.f;
    const float3 nn = entering ? n : neg3(n);
    const float eta = entering ? 1.f / ior : ior;

    // ---- stage 1: a direction about an axis --------------------------------------------------------
    const bool is_ct = tag == RRS_MAT_COOK_TORRANCE || tag == RRS_MAT_COOK_TORRANCE_REFRACT || tag == RRS_MAT_COOK_TORRANCE_GLASS;
    const float fres_p = schlick_scalar(m.m2.z, nv_s);  // Plastic: Fresnel-selected lobe (material.rs:575-579)
    const bool plastic_spec = tag == RRS_MAT_PLASTIC && u0 < fres_p;
    const bool beckmann = is_ct || plastic_spec;
    const bool cosine = tag == RRS_MAT_LAMBERTIAN || (tag == RRS_MAT_PLASTIC && !plastic_spec);
    float3 sd = f3(0, 0, 0);
    if (beckmann || cosine) {
        const float3 axis = tag == RRS_MAT_COOK_TORRANCE_REFRACT ? nn : n;  // CookTorranceGlass samples about the UNflipped normal
        const float ua = tag == RRS_MAT_PLASTIC ? u1 : u0, ub = tag == RRS_MAT_PLASTIC ? u2 : u1;
        float sint, cost, uphi;
        if (cosine) {  // Pdf::Cosine generate material.rs:982-993: (u, uphi) = (ua, ub)
            sint = sqrtf(ua);
            cost = sqrtf(1.f - ua);
            uphi = ub;
        } else {       // Beckmann half vector material.rs:1006-1020 / 1137-1161: (uphi, uxi) = (ua, ub)
            float tan2 = -alpha2 * logf(1.f - ub);
            cost = rsqrtf(1.f + tan2);
            sint = sqrtf(fmaxf(0.f, 1.f - cost * cost));
            uphi = ua;
        }
        float3 e1, e2;
        orthonormal_basis(axis, e1, e2);
        float sn, cs;
        sincospif(2.f * uphi, &sn, &cs);
        sd = add3(add3(scale3(e1, cs * sint), scale3(e2, sn * sint)), scale3(axis, cost));
    }

    // ---- stage 2: what this variant does with it -----------------------------------------------------
    enum { K_NONE, K_DIFFUSE, K_SPEC_REFLECT, K_SPEC_REFRACT, K_CT_REFLECT, K_CT_REFRACT };
    int kind = K_NONE;
    float3 about = n;         // the vector the ray is mirrored / refracted about
    bool reflect = false, refract = false;
    float3 rcolor = color;    // colour of the reflection lobe
    int fresnel_mode = 1;     // ct_reflection: 0 metallic r0, 1 dielectric Schlick, 2 cancelled by the caller's division
    float3 n_eval = n;        // normal the Cook-Torrance weight is evaluated with
    float div = 1.f;
    bool keep_one_minus_f = false;
    switch (tag) {
        case RRS_MAT_LAMBERTIAN:  // (color/pi * n.l) / (n.l/pi) == color
            kind = K_DIFFUSE;
            break;
        case RRS_MAT_REFLECT:
            kind = K_SPEC_REFLECT;
            reflect = true;
            break;
        case RRS_MAT_REFRACT:
            kind = K_SPEC_REFRACT;
            about = nn;
            refract = true;
            break;
        case RRS_MAT_GLASS: {
            const float sin2 = 1.f - nv_s * nv_s;
            bool do_reflect = eta * eta * sin2 >= 1.f;
            if (!do_reflect) do_reflect = u0 < schlick_scalar(m.m2.z, dot3(nn, v));
            about = nn;
            kind = do_reflect ? K_SPEC_REFLECT : K_SPEC_REFRACT;
            reflect = do_reflect;
            refract = !do_reflect;
            break;
        }
        case RRS_MAT_COOK_TORRANCE:
            kind = K_CT_REFLECT;
            about = sd;
            reflect = true;
            fresnel_mode = __float_as_uint(m.m2.y) == RRS_FRESNEL_METALLIC ? 0 : 1;
            break;
        case RRS_MAT_COOK_TORRANCE_REFRACT:
            kind = K_CT_REFRACT;
            about = entering ? sd : neg3(sd);
            refract = true;
            n_eval = nn;
            keep_one_minus_f = true;
            break;
        case RRS_MAT_COOK_TORRANCE_GLASS: {
            about = entering ? sd : neg3(sd);
            n_eval = nn;
            const float cos_t = dot3(about, v);
            const float sin2 = 1.f - cos_t * cos_t;
            if (eta * eta * sin2 >= 1.f) {  // total internal reflection: Fresnel kept, no division
                kind = K_CT_REFLECT;
                reflect = true;
            } else if (u2 < schlick_scalar(m.m2.z, cos_t)) {  // F / F cancels
                kind = K_CT_REFLECT;
                reflect = true;
                fresnel_mode = 2;
            } else {
                kind = K_CT_REFRACT;
                refract = true;
            }
            break;
        }
        case RRS_MAT_PLASTIC:
            if (plastic_spec) {
                kind = K_CT_REFLECT;
                about = sd;
                reflect = true;
                rcolor = xyz(m.m1);
                div = fres_p;
            } else {
                kind = K_DIFFUSE;
            }
            break;
        default:  // NoReflect material.rs:107
            break;
    }

    // ---- stage 3: the outgoing direction ---------------------------------------------------------------
    float3 l = sd;
    if (reflect) {
        l = reflect3(about, v);
    } else if (refract) {
        if (!refract3(about, v, eta, l)) return r;  // NoScatter
    }

    // ---- stage 4: the weight ---------------------------------------------------------------------------
    switch (kind) {
        case K_DIFFUSE:
            r.dir = l;
            r.color = color;
            r.scatter = true;
            return r;
        case K_SPEC_REFLECT: {  // color / |n.l| * (n.l)
            float nl = dot3(about, l);
            r.dir = l;
            r.color = scale3(color, nl / fabsf(nl));
            r.scatter = true;
            return r;
        }
        case K_SPEC_REFRACT:
            r.dir = l;
            r.color = dot3(l, v) > 0.f ? f3(0, 0, 0) : color;
            r.scatter = true;
            return r;
        case K_CT_REFLECT:
            return ct_reflection(m, rcolor, fresnel_mode, n_eval, about, v, l, div);
        case K_CT_REFRACT:
            return ct_refraction(m, color, n_eval, about, v, l, keep_one_minus_f);
        default:
            return r;
    }
}

template <bool STAGED>
__device__ __forceinline__ ScatterOut material_evaluate(const DMat& m, float3 n, float3 v, float u0, float u1, float u2) {
    return STAGED ? material_evaluate_staged(m, n, v, u0, u1, u2) : material_evaluate_cases(m, n, v, u0, u1, u2);
}

// Scene::background lib.rs:254-285.  Texels are float4 (rgb, -).  In f64 the bilinear
// weights are (ceil(x)-x, x-floor(x)); for non-integral x that is (1-fx, fx).  x is integral
// with probability ~0 in f64 but ~1e-4 in fp32, so the kernel always uses (1-fx, fx): that is
// what the f64 reference computes for the real-valued x an fp32-integral x stands for.
// Indices that the reference would panic on (theta == pi, phi == 2pi) are clamped.
// Texel coordinates of a direction (also the cell index of the environment's sampling table, env.cuh).
__device__ __forceinline__ void background_coords(const DScene& sc, float3 dir, float& x, float& y) {
    dir = normalize3(dir);
    float phi = atan2f(dir.z, dir.x) + RRS_PI_F;
    float theta = acosf(fminf(1.f, fmaxf(-1.f, dir.y)));
    x = phi * (0.5f / RRS_PI_F) * (float)(sc.hdri_w - 1);
    y = theta * (1.0f / RRS_PI_F) * (float)(sc.hdri_h - 1);
}

__device__ __forceinline__ float3 background(const DScene& sc, float3 dir) {
    float x, y;
    background_coords(sc, dir, x, y);
    float xf = floorf(x), yf = floorf(y);
    float fx = x - xf, fy = y - yf;
    uint32_t j = (uint32_t)xf, i = (uint32_t)yf;
    uint32_t j0 = min(j, sc.hdri_w - 1), j1 = min(j + 1, sc.hdri_w - 1);
    uint32_t i0 = min(i, sc.hdri_h - 1), i1 = min(i + 1, sc.hdri_h - 1);
    float4 f0 = __ldg(sc.hdri + (size_t)i0 * sc.hdri_w + j0);
    float4 f1 = __ldg(sc.hdri + (size_t)i1 * sc.hdri_w + j0);
    float4 f2 = __ldg(sc.hdri + (size_t)i0 * sc.hdri_w + j1);
    float4 f3_ = __ldg(sc.hdri + (size_t)i1 * sc.hdri_w + j1);
    float w0 = (1.f - fx) * (1.f - fy), w1 = (1.f - fx) * fy, w2 = fx * (1.f - fy), w3 = fx * fy;
    return f3(f0.x * w0 + f1.x * w1 + f2.x * w2 + f3_.x * w3, f0.y * w0 + f1.y * w1 + f2.y * w2 + f3_.y * w3,
              f0.z * w0 + f1.z * w1 + f2.z * w2 + f3_.z * w3);
}

// Geometric normal of primitive `p` at position `pos` (Hittable::normal: geometry.rs:134-136,
// 273-282, 377-379).
__device__ __forceinline__ float3 prim_normal(const DPrim* prims, uint32_t pi, float4 a, float3 pos) {
    uint32_t type = __float_as_uint(a.w) & 3u;
    const float4* pp = reinterpret_cast<const float4*>(prims + pi);
    if (type == RRS_SPHERE) return normalize3(sub3(pos, xyz(a)));
    float4 b = __ldg(pp + 1);
    if (type == RRS_PLANE) {
        uint32_t ax = __float_as_uint(b.z);
        float s = (ax & 1u) ? -1.f : 1.f;
        uint32_t k = ax >> 1;
        return f3(k == 0 ? s : 0.f, k == 1 ? s : 0.f, k == 2 ? s : 0.f);
    }
    float4 c = __ldg(pp + 2);
    float3 p1 = xyz(a);
    return normalize3(cross3(sub3(xyz(b), p1), sub3(xyz(c), p1)));  // Triangle::new geometry.rs:341-355
}

}  // namespace rrs
