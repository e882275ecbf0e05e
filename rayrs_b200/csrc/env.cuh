// Environment importance sampling for RRS_FLAG_ENV_SAMPLING: the sampling table of the HDRI, its density, and the
// two BSDF terms next-event estimation needs at a Lambertian or Cook-Torrance vertex.
//
// Table (built once per scene on the host, api.cu build_env_table): the (w-1) x (h-1) cells between texel centres of
// background()'s parametrisation, x = phi / 2pi * (w-1), y = theta / pi * (h-1).  A cell's weight is the largest
// max(|r|, |g|, |b|) of its 4 corner texels times its solid angle, so it is positive wherever the bilinear lookup can
// be non-zero.  A row is drawn from the marginal CDF, a cell from the row's conditional CDF, and the direction
// uniformly in solid angle inside the cell (phi uniform, cos theta uniform): the density is constant per cell.
// Both CDFs hold multiples of 2^-24 (and every positive cell at least one step), the resolution of the 24-bit
// uniforms that pick the cell: the probability of drawing a cell is then exactly its stored CDF step, and the density
// computed from the steps is the density the sampler realises.
#pragma once
#include "shading.cuh"

namespace rrs {

// origin word of a shadow ray (RRS_FLAG_ENV_SAMPLING): primitive index | RRS_SHADOW.  Bits 28..30 are free
// (RRS_PRIM_MASK, RRS_ORG64); a shadow ray never starts at the camera (RRS_NO_PRIM).
#define RRS_SHADOW 0x40000000u
// RNG slot of the environment draw at bounce b: existing slots are 0 (camera) and b + 1 <= 255 (bounce b)
#define RRS_ENV_SLOT 0x100u

struct DEnv {
    const float* marg;   // [ch] start of each row in the marginal CDF; nullptr: the map is black (nothing to sample)
    const float2* row;   // [ch] (cos theta at the row's top edge, cos theta top - cos theta bottom)
    const float* cond;   // [ch][cw] start of each cell in its row's conditional CDF
    float* wmis;         // [2][capacity] MIS weight of each queued continuation ray (the render's side array)
    uint32_t cw, ch;     // cells: hdri_w - 1, hdri_h - 1
    float inv_dphi;      // cw / 2pi
};

// largest k < n with a[k] <= u (a[0] == 0 <= u): lands on a cell of non-zero width
__device__ __forceinline__ uint32_t cdf_find(const float* __restrict__ a, uint32_t n, float u) {
    uint32_t lo = 0, hi = n;
    while (hi - lo > 1u) {
        const uint32_t mid = (lo + hi) >> 1;
        if (__ldg(a + mid) <= u) lo = mid;
        else hi = mid;
    }
    return lo;
}

__device__ __forceinline__ float cdf_step(const float* __restrict__ a, uint32_t n, uint32_t k) {
    return (k + 1u < n ? __ldg(a + k + 1u) : 1.f) - __ldg(a + k);  // exact: both ends are multiples of 2^-24
}

// solid-angle density of the cell (i, j)
__device__ __forceinline__ float env_cell_pdf(const DEnv& e, uint32_t i, uint32_t j) {
    const float pm = cdf_step(e.marg, e.ch, i);
    const float pc = cdf_step(e.cond + (size_t)i * e.cw, e.cw, j);
    return pm * pc * e.inv_dphi / __ldg(&e.row[i].y);
}

// density of direction `dir`, in the cell background() reads it from (same coordinates, bit for bit)
__device__ __forceinline__ float env_pdf(const DScene& sc, const DEnv& e, float3 dir) {
    if (e.marg == nullptr) return 0.f;
    float x, y;
    background_coords(sc, dir, x, y);
    const uint32_t j = min((uint32_t)floorf(x), e.cw - 1u), i = min((uint32_t)floorf(y), e.ch - 1u);
    return env_cell_pdf(e, i, j);
}

// Draw a direction.  (u0, u1) pick the row and the cell (24-bit uniforms, as the device RNG hands them out);
// (u0 + 2^-24 * lo0, u1 + 2^-24 * lo1) as 48-bit uniforms place the direction inside the cell, so that the position
// stays continuous even in a cell one CDF step wide.  Returns the density of the drawn cell: the density the sampler
// realises.  (env_pdf of the fp32 direction can read a neighbouring cell when the direction lies within rounding of
// the cell's edge, and a neighbour 10^6 times dimmer, or black, would turn the shadow ray's weight into a spike.)
__device__ __forceinline__ float env_sample(const DScene& sc, const DEnv& e, float u0, float u1, float lo0, float lo1,
                                            float3& dir) {
    const uint32_t i = cdf_find(e.marg, e.ch, u0);
    const float pm = cdf_step(e.marg, e.ch, i);
    const float* cond = e.cond + (size_t)i * e.cw;
    const uint32_t j = cdf_find(cond, e.cw, u1);
    const float pc = cdf_step(cond, e.cw, j);
    const float t0 = fminf(((u0 - __ldg(e.marg + i)) + lo0 * 0x1p-24f) / pm, 1.f);
    const float t1 = fminf(((u1 - __ldg(cond + j)) + lo1 * 0x1p-24f) / pc, 1.f);
    const float2 r = __ldg(&e.row[i]);
    const float cy = r.x - t0 * r.y;
    const float sy = sqrtf(fmaxf(0.f, (1.f - cy) * (1.f + cy)));
    float sp, cp;
    sincospif(2.f * ((float)j + t1) / (float)e.cw, &sp, &cp);
    dir = f3(-sy * cp, cy, -sy * sp);  // phi = atan2(z, x) + pi, theta = acos(y)
    return pm * pc * e.inv_dphi / r.y;  // env_cell_pdf(e, i, j)
}

// Beckmann D(h) for cos theta_h = nh, with tan^2 from |n x h|^2 (no cancellation at alpha = 0.01)
__device__ __forceinline__ float beckmann_d(float alpha2, float3 n, float3 h, float nh) {
    const float3 c = cross3(n, h);
    const float t = dot3(c, c) / (nh * nh * alpha2);
    if (!(t < 80.f)) return 0.f;  // e^-80: below every fp32 weight, and keeps 1 / cos^4 finite
    const float nh2 = nh * nh;
    return __expf(-t) / (RRS_PI_F * alpha2 * nh2 * nh2);
}

// What the plain render's estimator does with direction l at a Lambertian or Cook-Torrance vertex: W = its weight
// (throughput factor, material_evaluate's colour) and pdf = the density with which its sampling procedure produces l.
// K = W * pdf is the kernel the plain render integrates.  Cook-Torrance: the half vector is drawn with density
// D cos theta_h (the reference's pdf omits the cosine, SURVEY F2) and mirrored (Jacobian 1 / (4 h.l)); W, and every
// case in which the plain sample is dropped, follow ct_reflection.  pdf == 0: the plain render never produces l.
__device__ __forceinline__ float nee_bsdf(const DMat& m, uint32_t tag, float3 n, float3 v, float3 l, float3& W) {
    W = f3(0.f, 0.f, 0.f);
    if (tag == RRS_MAT_LAMBERTIAN) {
        const float nl = dot3(n, l);
        if (!(nl > 0.f)) return 0.f;
        W = xyz(m.m0);
        return nl * (1.f / RRS_PI_F);
    }
    float3 hh = add3(v, l);
    if (hh.x == 0.f && hh.y == 0.f && hh.z == 0.f) return 0.f;
    const float3 h = normalize3(hh);
    const float nh = dot3(n, h);
    const float hv = dot3(h, v);
    const float nl_s = dot3(n, l);
    const float nv = fabsf(dot3(n, v));
    if (!(nh > 0.f) || !(hv > 0.f) || nl_s <= 0.f || nv == 0.f) return 0.f;
    const float g = fminf(2.f * nh * nv / hv, fminf(2.f * nh * nl_s / hv, 1.f));
    const float3 F = fresnel_ct(m, __float_as_uint(m.m2.y) == RRS_FRESNEL_METALLIC, hv);
    W = scale3(mul3(xyz(m.m0), F), g * dot3(h, l) / nv);
    return beckmann_d(m.m1.w, n, h, nh) * nh / (4.f * hv);  // h.l == h.v for the mirrored direction
}

// Power-heuristic terms for densities a (this strategy) and b (the other), at least one of them positive:
// a^2 / (a^2 + b^2) and a b / (a^2 + b^2), through the ratio of the smaller to the larger so that no square overflows.
__device__ __forceinline__ float mis_power(float a, float b) {
    const float s = fminf(a, b) / fmaxf(a, b), s2 = s * s;
    return (a >= b ? 1.f : s2) / (1.f + s2);
}
__device__ __forceinline__ float mis_cross(float a, float b) {
    const float s = fminf(a, b) / fmaxf(a, b);
    return s / (1.f + s * s);
}

}  // namespace rrs
