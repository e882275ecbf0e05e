// rayrs oracle — CPU f64 restatement of the rayrs-lib path-tracing hot path.
//
// THIS IS TEST INFRASTRUCTURE, NOT PRODUCT CODE.  Only tests/, __graft_entry__.smoke()
// and bench.py's cpu_baseline / --impl reference legs may load it.  The product
// (rayrs_b200/csrc + rayrs_b200/host) never links, imports or calls anything here.
//
// What it restates (citations are /root/reference/<file>:<line>):
//   vecmath      rayrs-lib/src/vecmath.rs:341-352,513-760   (dot/cross/unit, reciprocal Div, basis)
//   geometry     rayrs-lib/src/geometry.rs:106-136 (sphere) 229-282 (plane) 341-379 (triangle)
//                458-513 (AABB slab) 544-550,577-582,640-645,674-733 (boxes)
//   bvh          rayrs-lib/src/bvh.rs:7-38 (SAH cost) 50-72 (update) 87-163 (BvhData)
//                227-317 (build_sah) 319-389 (build_midpoint) 391-415 (traverse)
//   material     rayrs-lib/src/material.rs:259-593 (scatter fns) 686-812 (evaluate_*)
//                913-1020 (Pdf) 1137-1161 (MicrofacetDistribution) 1233-1442 (brdf/btdf)
//                1472-1518 (schlick/reflect/refract) 1048-1084 (Emission)
//   integrator   rayrs-lib/src/lib.rs:99-133,202-210 (Camera) 254-285 (background) 521-560 (radiance)
//   tile loop    rayrs/src/main.rs:52-94 (16x16 tiles, F8 index mapping, pixel/spp)
//
// Pinning: the reference cannot be built here (no Rust toolchain).  The restatement is
// pinned against every numeric known-answer test the reference holds for this path
// (tests/test_oracle_kat.py lists them with file:line), and its camera / primary rays /
// pixel mapping / sphere-scene constants against the geometry of the six renders the
// reference ships (examples/*.png; tests/test_reference_images.py); its Midpoint build
// reproduces the expected dumps of the construction tests the reference carries commented
// out (bvh.rs:436-541).  Triangle intersection, BSDF values, radiance(), background() and the
// SAH tree shape are NOT pinned by any reference test or output ("parity unpinned" for
// those; see DESIGN.md).
//
// One deliberate deviation: rand::random::<f64>() (thread_rng, OS seeded, not
// reproducible; lib.rs:206-207,539 and material.rs call sites) is replaced by a
// counter-based Philox4x32-7 stream keyed by (seed; pixel, sample, slot) so that
// results are reproducible and can be sample-matched with the GPU backend.
//
// One addition that is not in the reference: the GPU backend's environment sampling (RRS_FLAG_ENV_SAMPLING), restated
// from rayrs_b200/csrc/api.cu build_env_table and env.cuh / wavefront.cu (EnvTable, env_sample, nee_bsdf, radiance with
// env; orc_render_env, orc_env_table, orc_env_sample, orc_env_pdf) so that ENV images can be sample-matched too.
// orc_render and radiance without it are unchanged.
//
// Build: see oracle/Makefile (g++ -O3 -ffp-contract=off: Rust never contracts a*b+c).

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <limits>
#include <memory>
#include <string>
#include <thread>
#include <vector>

namespace orc {

static const double PI = 3.14159265358979323846264338327950288;
static const double FRAC_1_PI = 0.318309886183790671537767526745028724;

// ------------------------------------------------------------------------------------
// vecmath.rs
// ------------------------------------------------------------------------------------
struct V3 {
    double x, y, z;
};
static inline V3 v3(double x, double y, double z) { return V3{x, y, z}; }
static inline V3 operator+(V3 a, V3 b) { return V3{a.x + b.x, a.y + b.y, a.z + b.z}; }
static inline V3 operator-(V3 a, V3 b) { return V3{a.x - b.x, a.y - b.y, a.z - b.z}; }
static inline V3 operator*(V3 a, V3 b) { return V3{a.x * b.x, a.y * b.y, a.z * b.z}; }
static inline V3 operator*(V3 a, double s) { return V3{a.x * s, a.y * s, a.z * s}; }
static inline V3 operator*(double s, V3 a) { return V3{s * a.x, s * a.y, s * a.z}; }
// vecmath.rs:690-698  Div<f64> multiplies by the reciprocal.
static inline V3 operator/(V3 a, double s) {
    double inv = 1. / s;
    return a * inv;
}
// vecmath.rs:533-535
static inline double dot(V3 a, V3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
// vecmath.rs:565-573
static inline V3 cross(V3 a, V3 b) {
    return V3{a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x};
}
static inline double mag2(V3 a) { return dot(a, a); }
static inline double mag(V3 a) { return std::sqrt(mag2(a)); }
// vecmath.rs:525-527
static inline V3 unit(V3 a) { return a / mag(a); }
static inline bool is_zeros(V3 a) { return a.x == 0. && a.y == 0. && a.z == 0.; }
// Rust f64::max/min return the non-NaN operand == C fmax/fmin.
static inline double rmax(double a, double b) { return std::fmax(a, b); }
static inline double rmin(double a, double b) { return std::fmin(a, b); }
// compiler-rt __powidf2 sequence for n=4 and n=5.
static inline double powi4(double a) {
    double a2 = a * a;
    return a2 * a2;
}
static inline double powi5(double a) {
    double a2 = a * a;
    double a4 = a2 * a2;
    return a * a4;
}
// vecmath.rs:341-352
static inline void orthonormal_basis(V3 n, V3& e1, V3& e2) {
    if (std::fabs(n.x) > std::fabs(n.y))
        e1 = unit(v3(n.z, 0., -n.x));
    else
        e1 = unit(v3(0., n.z, -n.y));
    e2 = unit(cross(n, e1));
}

struct Ray {
    V3 o, d;
    // lib.rs:41-43
    V3 point(double t) const { return o + d * t; }
};

// ------------------------------------------------------------------------------------
// RNG: Philox4x32 (Salmon et al., SC'11; Random123 reference constants), kPhiloxRounds = 7 rounds for the render
// stream — the smallest round count the paper reports as passing BigCrush, and what the GPU backend draws; orc_philox
// exposes the round count so that both 7 and 10 are pinned on Random123's published known answers.
// counter = (pixel, sample, slot, block), key = (seed_lo, seed_hi).
// slot 0: camera jitter (word0 -> x, word1 -> y).  slot b+1: bounce b, words 0..2 are the
// material's draws in call order, word 3 is the Russian-roulette draw.
// ------------------------------------------------------------------------------------
static const int kPhiloxRounds = 7;
static inline void philox4x32(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0,
                              uint32_t k1, uint32_t out[4], int rounds = kPhiloxRounds) {
    const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
    for (int r = 0; r < rounds; ++r) {
        uint64_t p0 = (uint64_t)M0 * c0;
        uint64_t p1 = (uint64_t)M1 * c2;
        uint32_t hi0 = (uint32_t)(p0 >> 32), lo0 = (uint32_t)p0;
        uint32_t hi1 = (uint32_t)(p1 >> 32), lo1 = (uint32_t)p1;
        uint32_t n0 = hi1 ^ c1 ^ k0;
        uint32_t n1 = lo1;
        uint32_t n2 = hi0 ^ c3 ^ k1;
        uint32_t n3 = lo0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += W0; k1 += W1;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

struct Rng {
    // mode 1: u = (w >> 8) * 2^-24  — the exact values the GPU backend uses (sample-matched).
    // mode 0: 53-bit uniforms from two Philox blocks (rand 0.7.3 resolution).
    uint64_t seed;
    uint32_t pixel, sample;
    int mode;
    double u[4];
    void load(uint32_t slot) {
        uint32_t a[4];
        philox4x32(pixel, sample, slot, 0u, (uint32_t)seed, (uint32_t)(seed >> 32), a);
        if (mode == 1) {
            for (int i = 0; i < 4; ++i) u[i] = (double)(a[i] >> 8) * (1.0 / 16777216.0);
        } else {
            uint32_t b[4];
            philox4x32(pixel, sample, slot, 1u, (uint32_t)seed, (uint32_t)(seed >> 32), b);
            for (int i = 0; i < 4; ++i) {
                uint64_t hi = a[i] >> 5, lo = b[i] >> 6;
                u[i] = ((double)hi * 67108864.0 + (double)lo) * (1.0 / 9007199254740992.0);
            }
        }
    }
};

// ------------------------------------------------------------------------------------
// geometry.rs
// ------------------------------------------------------------------------------------
struct AABB {
    double xmin, xmax, ymin, ymax, zmin, zmax;
    // geometry.rs:458-513
    bool intersect(const Ray& ray, double tmin, double tmax) const {
        {
            double hi = xmax - ray.o.x, lo = xmin - ray.o.x, inv = 1. / ray.d.x;
            double t0, t1;
            if (inv < 0.) { t0 = hi * inv; t1 = lo * inv; } else { t0 = lo * inv; t1 = hi * inv; }
            tmin = rmax(tmin, t0);
            tmax = rmin(tmax, t1);
            if (tmax <= tmin) return false;
        }
        {
            double hi = ymax - ray.o.y, lo = ymin - ray.o.y, inv = 1. / ray.d.y;
            double t0, t1;
            if (inv < 0.) { t0 = hi * inv; t1 = lo * inv; } else { t0 = lo * inv; t1 = hi * inv; }
            tmin = rmax(tmin, t0);
            tmax = rmin(tmax, t1);
            if (tmax <= tmin) return false;
        }
        {
            double hi = zmax - ray.o.z, lo = zmin - ray.o.z, inv = 1. / ray.d.z;
            double t0, t1;
            if (inv < 0.) { t0 = hi * inv; t1 = lo * inv; } else { t0 = lo * inv; t1 = hi * inv; }
            tmin = rmax(tmin, t0);
            tmax = rmin(tmax, t1);
            if (tmax <= tmin) return false;
        }
        return true;
    }
    // geometry.rs:577-582
    V3 center() const {
        return v3((xmax - xmin) / 2. + xmin, (ymax - ymin) / 2. + ymin, (zmax - zmin) / 2. + zmin);
    }
    // geometry.rs:609-613
    double volume() const { return (xmax - xmin) * (ymax - ymin) * (zmax - zmin); }
    // geometry.rs:640-645
    double surface_area() const {
        double x = xmax - xmin, y = ymax - ymin, z = zmax - zmin;
        return 2. * x * y + 2. * y * z + 2. * x * z;
    }
    // geometry.rs:674-683
    AABB expand(const AABB& o) const {
        return AABB{rmin(xmin, o.xmin), rmax(xmax, o.xmax), rmin(ymin, o.ymin),
                    rmax(ymax, o.ymax), rmin(zmin, o.zmin), rmax(zmax, o.zmax)};
    }
};

enum Axis { AX_X = 0, AX_XREV = 1, AX_Y = 2, AX_YREV = 3, AX_Z = 4, AX_ZREV = 5 };

struct DrawSrc {
    // hands out the material draws of one bounce in call order (words 0..2; a fourth for Plastic's diffuse lobe under a caller's pdf)
    const double* u;
    int next;
    double draw() { return u[next++]; }
};

// trait Hittable, geometry.rs:15-38.  area + sample serve Pdf::Hittable only (material.rs:943-950,1027), which
// radiance() never reaches because it passes pdf=None (lib.rs:532); they are restated for the dormant
// next-event-estimation hook, material_evaluate(..., light) below.
struct Hittable {
    virtual ~Hittable() {}
    virtual bool intersect(const Ray& ray, double& t) const = 0;
    virtual V3 normal(V3 p) const = 0;
    virtual AABB bbox() const = 0;
    virtual double area() const = 0;
    virtual V3 sample(DrawSrc& rs) const = 0;
};

struct Sphere final : Hittable {
    double radius2;
    V3 origin;
    Sphere(double r, V3 o) : radius2(r * r), origin(o) {}
    // geometry.rs:106-132
    bool intersect(const Ray& ray, double& t) const override {
        V3 od = ray.o - origin;
        double a = mag2(ray.d);
        double b = 2. * dot(ray.d, od);
        double c = mag2(od) - radius2;
        double desc = b * b - 4. * a * c;
        if (desc > 0.) {
            double t1 = (-b - std::sqrt(desc)) / (2. * a);
            double t2 = (-b + std::sqrt(desc)) / (2. * a);
            if (t1 < 0.) {
                if (t2 < 0.) return false;
                t = t2;
                return true;
            }
            t = t1;
            return true;
        }
        return false;
    }
    V3 normal(V3 p) const override { return unit(p - origin); }
    // geometry.rs:138-140
    double area() const override { return 4. * PI * radius2; }
    // geometry.rs:142-152 ("FIXME: This is not uniform on the unit sphere..." — restated as written)
    V3 sample(DrawSrc& rs) const override {
        double u = rs.draw();
        double phi = 2. * PI * rs.draw();
        double x = std::cos(phi) * 2. * std::sqrt(u * (1. - u));
        double y = std::sin(phi) * 2. * std::sqrt(u * (1. - u));
        double z = 1. - 2. * u;
        return v3(x, y, z) * std::sqrt(radius2) + origin;
    }
    // geometry.rs:687-696
    AABB bbox() const override {
        double r = std::sqrt(radius2);
        return AABB{origin.x - r, origin.x + r, origin.y - r, origin.y + r, origin.z - r, origin.z + r};
    }
};

struct Plane final : Hittable {
    int axis;
    double umin, umax, vmin, vmax, pos;
    Plane(int ax, double u0, double u1, double v0, double v1, double p)
        : axis(ax), umin(u0), umax(u1), vmin(v0), vmax(v1), pos(p) {}
    // Range::contains is half-open [start, end).
    static bool contains(double lo, double hi, double v) { return lo <= v && v < hi; }
    // geometry.rs:229-271
    bool intersect(const Ray& ray, double& t) const override {
        switch (axis) {
            case AX_X: case AX_XREV:
                if (ray.d.x != 0.) {
                    double tt = (pos - ray.o.x) / ray.d.x;
                    V3 p = ray.point(tt);
                    if (contains(umin, umax, p.y) && contains(vmin, vmax, p.z)) { t = tt; return true; }
                }
                return false;
            case AX_Y: case AX_YREV:
                if (ray.d.y != 0.) {
                    double tt = (pos - ray.o.y) / ray.d.y;
                    V3 p = ray.point(tt);
                    if (contains(umin, umax, p.x) && contains(vmin, vmax, p.z)) { t = tt; return true; }
                }
                return false;
            default:
                if (ray.d.z != 0.) {
                    double tt = (pos - ray.o.z) / ray.d.z;
                    V3 p = ray.point(tt);
                    if (contains(umin, umax, p.x) && contains(vmin, vmax, p.y)) { t = tt; return true; }
                }
                return false;
        }
    }
    // geometry.rs:273-282
    V3 normal(V3) const override {
        switch (axis) {
            case AX_X: return v3(1., 0., 0.);
            case AX_XREV: return v3(-1., 0., 0.);
            case AX_Y: return v3(0., 1., 0.);
            case AX_YREV: return v3(0., -1., 0.);
            case AX_Z: return v3(0., 0., 1.);
            default: return v3(0., 0., -1.);
        }
    }
    // geometry.rs:284-286
    double area() const override { return (umax - umin) * (vmax - vmin); }
    // geometry.rs:288-299
    V3 sample(DrawSrc& rs) const override {
        double u = rs.draw() * (umax - umin) + umin;
        double v = rs.draw() * (vmax - vmin) + vmin;
        switch (axis) {
            case AX_X: case AX_XREV: return v3(pos, u, v);
            case AX_Y: case AX_YREV: return v3(u, pos, v);
            default: return v3(u, v, pos);
        }
    }
    // geometry.rs:699-718
    AABB bbox() const override {
        switch (axis) {
            case AX_X: case AX_XREV: return AABB{pos, pos, umin, umax, vmin, vmax};
            case AX_Y: case AX_YREV: return AABB{umin, umax, pos, pos, vmin, vmax};
            default: return AABB{umin, umax, vmin, vmax, pos, pos};
        }
    }
};

struct Triangle final : Hittable {
    V3 p1, p2, p3, e1, e2, n;
    double tri_area;
    // geometry.rs:341-355
    Triangle(V3 a, V3 b, V3 c) : p1(a), p2(b), p3(c) {
        e1 = p2 - p1;
        e2 = p3 - p1;
        V3 nn = cross(e1, e2);
        n = unit(nn);
        tri_area = mag(nn) / 2.;
    }
    // geometry.rs:359-375
    bool intersect(const Ray& ray, double& t) const override {
        V3 T = ray.o - p1;
        V3 P = cross(ray.d, e2);
        V3 Q = cross(T, e1);
        double den = dot(P, e1);
        double d = dot(Q, e2) / den;
        double u = dot(P, T) / den;
        double v = dot(Q, ray.d) / den;
        if (d < 0. || u < 0. || v < 0. || u + v > 1.) return false;
        t = d;
        return true;
    }
    V3 normal(V3) const override { return n; }
    // geometry.rs:381-383 (area = |e1 x e2| / 2, set by Triangle::new)
    double area() const override { return tri_area; }
    // geometry.rs:385-387: the reference's stub returns the origin and draws nothing
    V3 sample(DrawSrc&) const override { return v3(0., 0., 0.); }
    // geometry.rs:721-733
    AABB bbox() const override {
        return AABB{rmin(p1.x, rmin(p2.x, p3.x)), rmax(p1.x, rmax(p2.x, p3.x)),
                    rmin(p1.y, rmin(p2.y, p3.y)), rmax(p1.y, rmax(p2.y, p3.y)),
                    rmin(p1.z, rmin(p2.z, p3.z)), rmax(p1.z, rmax(p2.z, p3.z))};
    }
};

// ------------------------------------------------------------------------------------
// material.rs
// ------------------------------------------------------------------------------------
enum MatTag {
    MAT_LAMBERTIAN = 0, MAT_REFLECT = 1, MAT_REFRACT = 2, MAT_GLASS = 3, MAT_COOK_TORRANCE = 4,
    MAT_CT_REFRACT = 5, MAT_CT_GLASS = 6, MAT_PLASTIC = 7, MAT_NO_REFLECT = 8
};
enum FresnelKind { FRESNEL_DIELECTRIC = 0, FRESNEL_METALLIC = 1 };

// Flat material record (mirrors the 12-double row the Python side passes):
//  [0] tag  [1..3] color  [4] alpha  [5] ior  [6] fresnel kind  [7..9] r0 (metallic) or
//  spec_color (plastic)
struct Material {
    int tag;
    V3 color;
    double alpha2;
    double ior;
    int fresnel_kind;
    V3 r0;    // SchlickMetallic(r0)
    V3 spec;  // Plastic spec_color
};

struct Emission {
    bool dark;
    double strength;
    V3 color;
    // material.rs:1077-1084
    V3 emit() const { return dark ? v3(0., 0., 0.) : strength * color; }
};

struct ScatterEvent {
    bool scatter;
    V3 color;
    Ray ray;
};
static inline ScatterEvent no_scatter() { return ScatterEvent{false, v3(0, 0, 0), Ray{v3(0, 0, 0), v3(0, 0, 0)}}; }

enum Direction { ENTERING = 0, EXITING = 1 };
// material.rs:1198-1231
static inline double dir_ior_ratio(Direction d, double ior) { return d == ENTERING ? 1. / ior : ior; }
static inline V3 dir_normal(Direction d, V3 n) { return d == ENTERING ? n : -1. * n; }
static inline void dir_iors(Direction d, double ior, double& curr, double& nw) {
    if (d == ENTERING) { curr = 1.; nw = ior; } else { curr = ior; nw = 1.; }
}

// material.rs:1472-1479
static inline double schlick_scalar(double ior_curr, double ior_new, V3 n, V3 v) {
    double r0 = (ior_curr - ior_new) / (ior_curr + ior_new);
    r0 = r0 * r0;
    return r0 + (1. - r0) * powi5(1. - dot(n, v));
}
// material.rs:1484-1489
static inline V3 schlick_vec(V3 r0, V3 n, V3 v) {
    return r0 + (v3(1., 1., 1.) - r0) * powi5(1. - dot(n, v));
}
// material.rs:1492-1496
static inline V3 reflect(V3 n, V3 v) { return 2. * dot(v, n) * n - v; }
// material.rs:1502-1518
static inline bool refract(V3 n, V3 v, double ior_ratio, V3& out) {
    double cos_theta = dot(v, n);
    double sin_theta = std::sqrt(1. - cos_theta * cos_theta);
    if (ior_ratio * sin_theta > 1.) return false;
    V3 par = ior_ratio * (cos_theta * n - v);
    V3 perp = -std::sqrt(1. - mag2(par)) * n;
    out = perp + par;
    return true;
}

// Fresnel::value material.rs:1457-1468
static inline V3 fresnel_value(const Material& m, int kind, V3 n, V3 v, Direction d) {
    if (kind == FRESNEL_DIELECTRIC) {
        double c, w;
        dir_iors(d, m.ior, c, w);
        double f = schlick_scalar(c, w, n, v);
        return v3(f, f, f);
    }
    return schlick_vec(m.r0, n, v);
}

// Pdf::Cosine generate material.rs:982-993
static inline V3 cosine_generate(V3 n, DrawSrc& rs) {
    V3 e1, e2;
    orthonormal_basis(n, e1, e2);
    double u = rs.draw();
    double phi = 2. * PI * rs.draw();
    double x = std::cos(phi) * std::sqrt(u);
    double y = std::sin(phi) * std::sqrt(u);
    double z = std::sqrt(1. - u);
    return x * e1 + y * e2 + z * n;
}

// Pdf::Beckmann generate material.rs:1006-1020 and MicrofacetDistribution::generate :1137-1161
static inline V3 beckmann_generate(double alpha2, V3 n, DrawSrc& rs, double* pdf_value) {
    V3 e1, e2;
    orthonormal_basis(n, e1, e2);
    double phi = 2. * PI * rs.draw();
    double tan2theta = -alpha2 * std::log(1. - rs.draw());
    double costheta = 1.0 / std::sqrt(1.0 + tan2theta);
    double sintheta = std::sqrt(1.0 - costheta * costheta);
    double x = std::cos(phi) * sintheta;
    double y = std::sin(phi) * sintheta;
    V3 h = x * e1 + y * e2 + costheta * n;
    if (pdf_value) {
        double nh = dot(n, h);
        *pdf_value = std::exp(-tan2theta / alpha2) / (PI * alpha2 * powi4(nh));
    }
    return h;
}

// Pdf::Beckmann(alpha2, Reflect).value material.rs:915-941
static inline double beckmann_pdf_value_reflect(double alpha2, V3 n, V3 l, V3 v) {
    V3 h = l + v;
    if (is_zeros(h)) return 1.;
    h = unit(h);
    double nh = std::fabs(dot(n, h));
    double theta_h = std::acos(nh);
    double tan_theta_h = std::tan(theta_h);
    if (std::isinf(tan_theta_h)) return 1.;
    return std::exp(-tan_theta_h * tan_theta_h / alpha2) / (PI * alpha2 * powi4(nh));
}

// Brdf for CookTorrance material.rs:1276-1322
static inline V3 ct_brdf(const Material& m, int fresnel_kind, V3 color, V3 n, V3 l, V3 v) {
    double nv = std::fabs(dot(n, v));
    double nl = std::fabs(dot(n, l));
    V3 h = v + l;
    if (nv == 0.0 || nl == 0.0) return v3(0, 0, 0);
    if (is_zeros(h)) return v3(0, 0, 0);
    h = unit(h);
    double nh = dot(n, h);
    double theta_h = std::acos(nh);
    double tan_theta_h = std::tan(theta_h);
    if (std::isinf(tan_theta_h)) return v3(0, 0, 0);
    double beckmann = std::exp(-tan_theta_h * tan_theta_h / m.alpha2) / (PI * m.alpha2 * powi4(nh));
    double hv = dot(h, v);
    double g = rmin(2.0 * nh * nv / hv, rmin(2.0 * nh * nl / hv, 1.));
    return color * fresnel_value(m, fresnel_kind, h, v, ENTERING) * beckmann * g / (4.0 * nv * nl);
}

// Btdf for CookTorrance material.rs:1362-1442
static inline V3 ct_btdf(const Material& m, V3 color, V3 n, V3 l, V3 v, Direction d) {
    double nv = std::fabs(dot(n, v));
    double nl = std::fabs(dot(n, l));
    double ior_ratio = dir_ior_ratio(d, m.ior);
    V3 h = ior_ratio > 1. ? l + ior_ratio * v : (-ior_ratio) * v - l;
    if (nv == 0.0 || nl == 0.0) return v3(0, 0, 0);
    if (is_zeros(h)) return v3(0, 0, 0);
    h = unit(h);
    double nh = dot(n, h);
    double theta_h = std::acos(nh);
    double tan_theta_h = std::tan(theta_h);
    if (std::isinf(tan_theta_h)) return v3(0, 0, 0);
    double beckmann = std::exp(-tan_theta_h * tan_theta_h / m.alpha2) / (PI * m.alpha2 * powi4(nh));
    double hl = std::fabs(dot(h, l));
    double hv = std::fabs(dot(h, v));
    double g = rmin(2.0 * nh * nv / hv, rmin(2.0 * nh * nl / hv, 1.));
    double denom = ior_ratio * hv + hl;
    denom = denom * denom;
    double norm_fac = hv * hl / (nv * nl);
    V3 fresnel = fresnel_value(m, FRESNEL_DIELECTRIC, h, v, d);
    return color * (v3(1, 1, 1) - fresnel) * beckmann * g * norm_fac * ior_ratio * ior_ratio / denom;
}

// CookTorrance::evaluate_reflection material.rs:721-758
static inline ScatterEvent ct_evaluate_reflection(const Material& m, int fresnel_kind, V3 color,
                                                  V3 position, V3 n, V3 h, V3 v, V3 l, double pdf) {
    if (dot(h, v) < 0.) return no_scatter();
    double nl = dot(n, l);
    if (nl < 0.0) return no_scatter();
    double frac_dwh_dwi = 4.0 * dot(h, l);
    V3 c = ct_brdf(m, fresnel_kind, color, n, l, v) * nl;
    c = c / pdf * frac_dwh_dwi;
    if (is_zeros(c)) return no_scatter();
    return ScatterEvent{true, c, Ray{position, l}};
}

// CookTorrance::evaluate_refraction material.rs:764-812
static inline ScatterEvent ct_evaluate_refraction(const Material& m, V3 color, V3 position, V3 n,
                                                  V3 h, V3 v, V3 l, double pdf, Direction d,
                                                  double ior_ratio) {
    if (dot(h, v) < 0.) return no_scatter();
    double nl = dot(n, l);
    if (nl > 0.0) return no_scatter();
    double hl = std::fabs(dot(h, l));
    double hv = std::fabs(dot(h, v));
    double denom = ior_ratio * hv + hl;
    denom = denom * denom;
    double dwh_dwi = hl / denom;
    V3 c = ct_btdf(m, color, n, l, v, d) * std::fabs(nl) / (ior_ratio * ior_ratio);
    c = c / (pdf * dwh_dwi);
    if (is_zeros(c)) return no_scatter();
    return ScatterEvent{true, c, Ray{position, l}};
}

// LambertianDiffuse::scatter with pdf=None material.rs:259-281
static inline ScatterEvent lambert_scatter(V3 color, V3 position, V3 n, DrawSrc& rs) {
    V3 l = cosine_generate(n, rs);
    V3 brdf = color * FRAC_1_PI;             // :1233-1243
    double pdfv = dot(n, l) * FRAC_1_PI;     // :913
    V3 c = brdf * dot(n, l) / pdfv;
    return ScatterEvent{true, c, Ray{position, l}};
}

// Pdf::Hittable value / generate, material.rs:943-950 and :1027 — the caller's pdf of the dormant next-event-estimation hook
static inline double pdf_hittable_value(const Hittable& g, V3 position, V3 n, V3 l) {
    Ray ray{position, l};
    double t;
    if (g.intersect(ray, t)) return mag2(position - ray.point(t)) / (dot(n, l) * g.area());
    return 0.;
}
static inline V3 pdf_hittable_generate(const Hittable& g, V3 position, DrawSrc& rs) { return unit(g.sample(rs) - position); }

// LambertianDiffuse::scatter with pdf=Some(Pdf::Hittable(light)) material.rs:259-281: the lobe is sampled from and weighted with
// Pdf::Mix(MixKind::Constant(0.5), pdf, Pdf::Cosine) — generate :1028-1034 (one draw picks the side), value :951-959
// (INFINITY below the surface, else the blend of the two densities).
static inline ScatterEvent lambert_scatter_mix(V3 color, V3 position, V3 n, const Hittable& light, DrawSrc& rs) {
    const double factor = 0.5;  // MixKind::Constant(0.5).value, material.rs:1529-1534
    V3 l = rs.draw() < factor ? pdf_hittable_generate(light, position, rs) : cosine_generate(n, rs);
    double pdfv;
    if (dot(n, l) < 0.) pdfv = std::numeric_limits<double>::infinity();
    else pdfv = factor * pdf_hittable_value(light, position, n, l) + (1. - factor) * (dot(n, l) * FRAC_1_PI);
    V3 brdf = color * FRAC_1_PI;  // :1233-1243
    V3 c = brdf * dot(n, l) / pdfv;
    return ScatterEvent{true, c, Ray{position, l}};
}

// CookTorrance::scatter material.rs:403-424
static inline ScatterEvent ct_scatter(const Material& m, int fresnel_kind, V3 color, V3 position,
                                      V3 n, V3 v, DrawSrc& rs) {
    V3 h = beckmann_generate(m.alpha2, n, rs, nullptr);
    V3 l = reflect(h, v);
    return ct_evaluate_reflection(m, fresnel_kind, color, position, n, h, v, l,
                                  beckmann_pdf_value_reflect(m.alpha2, n, l, v));
}

// Material::evaluate material.rs:91-109.  radiance() always passes pdf = None (lib.rs:532): light == nullptr.  A caller's
// pdf (light != nullptr: Pdf::Hittable(light)) is handed to every Bsdf::scatter, and only LambertianDiffuse::scatter
// — reached directly or as Plastic's diffuse lobe — looks at it; every other arm names its parameter `_pdf`.
static ScatterEvent material_evaluate(const Material& m, V3 position, V3 normal, V3 view, DrawSrc& rs,
                                      const Hittable* light = nullptr) {
    switch (m.tag) {
        case MAT_LAMBERTIAN:
            if (light) return lambert_scatter_mix(m.color, position, normal, *light, rs);
            return lambert_scatter(m.color, position, normal, rs);
        case MAT_REFLECT: {  // material.rs:283-303
            V3 l = reflect(normal, view);
            V3 brdf = m.color / std::fabs(dot(normal, l));  // :1254-1266
            V3 c = brdf * dot(normal, l) / 1.;               // Pdf::Dirac value = 1
            return ScatterEvent{true, c, Ray{position, l}};
        }
        case MAT_REFRACT: {  // material.rs:305-337
            double cos_theta = dot(normal, view);
            Direction d = cos_theta > 0. ? ENTERING : EXITING;
            V3 n = dir_normal(d, normal);
            V3 l;
            if (!refract(n, view, dir_ior_ratio(d, m.ior), l)) return no_scatter();
            V3 btdf = dot(l, view) > 0. ? v3(0, 0, 0) : m.color / std::fabs(dot(n, l));  // :1333-1351
            V3 c = btdf * std::fabs(dot(n, l)) / 1.;
            return ScatterEvent{true, c, Ray{position, l}};
        }
        case MAT_GLASS: {  // material.rs:339-401
            double cos_theta = dot(normal, view);
            Direction d = cos_theta > 0. ? ENTERING : EXITING;
            V3 n = dir_normal(d, normal);
            double sin2theta = 1. - cos_theta * cos_theta;
            double ior_ratio = dir_ior_ratio(d, m.ior);
            if (ior_ratio * ior_ratio * sin2theta >= 1.) {
                V3 l = reflect(n, view);
                V3 c = (m.color / std::fabs(dot(n, l))) * dot(n, l);
                return ScatterEvent{true, c, Ray{position, l}};
            }
            double ic, in;
            dir_iors(d, m.ior, ic, in);
            double fresnel = schlick_scalar(ic, in, n, view);
            if (rs.draw() < fresnel) {
                V3 l = reflect(n, view);
                V3 c = (m.color / std::fabs(dot(n, l))) * dot(n, l);
                return ScatterEvent{true, c, Ray{position, l}};
            }
            V3 l;
            bool ok = refract(n, view, ior_ratio, l);
            if (!ok) return no_scatter();  // the reference unwrap()s; unreachable up to rounding
            V3 btdf = dot(l, view) > 0. ? v3(0, 0, 0) : m.color / std::fabs(dot(n, l));
            V3 c = btdf * std::fabs(dot(n, l));
            return ScatterEvent{true, c, Ray{position, l}};
        }
        case MAT_COOK_TORRANCE:
            return ct_scatter(m, m.fresnel_kind, m.color, position, normal, view, rs);
        case MAT_CT_REFRACT: {  // material.rs:426-467
            Direction d = dot(normal, view) > 0. ? ENTERING : EXITING;
            V3 n = dir_normal(d, normal);
            double ior_ratio = dir_ior_ratio(d, m.ior);
            double pdfv;
            V3 h = beckmann_generate(m.alpha2, n, rs, &pdfv);
            h = dir_normal(d, h);
            V3 l;
            if (!refract(h, view, ior_ratio, l)) return no_scatter();
            return ct_evaluate_refraction(m, m.color, position, n, h, view, l, pdfv, d, ior_ratio);
        }
        case MAT_CT_GLASS: {  // material.rs:469-565
            double pdfv;
            V3 h = beckmann_generate(m.alpha2, normal, rs, &pdfv);
            Direction d = dot(normal, view) > 0. ? ENTERING : EXITING;
            h = dir_normal(d, h);
            V3 n = dir_normal(d, normal);
            double cos_theta = dot(h, view);
            double ior_ratio = dir_ior_ratio(d, m.ior);
            double sin2_theta = 1. - cos_theta * cos_theta;
            if (ior_ratio * ior_ratio * sin2_theta >= 1.) {
                V3 l = reflect(h, view);
                return ct_evaluate_reflection(m, FRESNEL_DIELECTRIC, m.color, position, n, h, view, l, pdfv);
            }
            double ic, in;
            dir_iors(d, m.ior, ic, in);
            double fresnel = schlick_scalar(ic, in, h, view);
            if (rs.draw() < fresnel) {
                V3 l = reflect(h, view);
                ScatterEvent e = ct_evaluate_reflection(m, FRESNEL_DIELECTRIC, m.color, position, n, h, view, l, pdfv);
                if (e.scatter) e.color = e.color / fresnel;
                return e;
            }
            V3 l;
            if (!refract(h, view, ior_ratio, l)) return no_scatter();  // reference expect()s
            ScatterEvent e = ct_evaluate_refraction(m, m.color, position, n, h, view, l, pdfv, d, ior_ratio);
            if (e.scatter) e.color = e.color / (1. - fresnel);
            return e;
        }
        case MAT_PLASTIC: {  // material.rs:567-593
            double fresnel = schlick_scalar(1., m.ior, normal, view);
            if (rs.draw() < fresnel) {
                ScatterEvent e = ct_scatter(m, FRESNEL_DIELECTRIC, m.spec, position, normal, view, rs);
                if (e.scatter) e.color = e.color / fresnel;
                return e;
            }
            if (light) return lambert_scatter_mix(m.color, position, normal, *light, rs);  // :588 forwards the pdf
            return lambert_scatter(m.color, position, normal, rs);
        }
        default:
            return no_scatter();  // NoReflect material.rs:107
    }
}

// ------------------------------------------------------------------------------------
// Object / Scene (lib.rs:213-245,298-512)
// ------------------------------------------------------------------------------------
struct Object {
    std::unique_ptr<Hittable> geom;
    int mat;       // index into Scene::materials
    int emission;  // index into Scene::emissions, -1 = Dark
    int id;        // index in the Vec<Object> handed to Scene::new (parity ID)
    AABB bbox() const { return geom->bbox(); }
};

// ------------------------------------------------------------------------------------
// bvh.rs
// ------------------------------------------------------------------------------------
struct BvhTree {
    bool leaf;
    AABB box;                                        // Node only
    std::vector<std::unique_ptr<BvhTree>> children;  // Node only
    const Object* obj;                               // LeafNode only
};

struct Hit {
    bool hit;
    double t;
    const Object* obj;
};

// RayIntersection::update bvh.rs:50-72
static inline Hit hit_update(Hit self, Hit other, double tmin) {
    if (!self.hit) return other;
    if (!other.hit) return self;
    if (other.t > tmin && other.t < self.t) return other;
    return self;
}

// BvhTree::intersect bvh.rs:391-415
static Hit tree_intersect(const BvhTree* n, const Ray& ray, double tmin, double tmax) {
    if (!n->leaf) {
        if (n->box.intersect(ray, tmin, tmax)) {
            Hit acc{false, 0., nullptr};
            for (const auto& ch : n->children) acc = hit_update(acc, tree_intersect(ch.get(), ray, tmin, tmax), tmin);
            return acc;
        }
        return Hit{false, 0., nullptr};
    }
    double t;
    if (n->obj->geom->intersect(ray, t)) {
        if (t > tmin && t < tmax) return Hit{true, t, n->obj};
    }
    return Hit{false, 0., nullptr};
}

static AABB bbox_of(const std::vector<const Object*>& objs, size_t lo, size_t hi) {
    // AxisAlignedBoundingBox::from_object_list geometry.rs:544-550
    AABB b = objs[lo]->bbox();
    for (size_t i = lo + 1; i < hi; ++i) b = b.expand(objs[i]->bbox());
    return b;
}

static inline double axis_of(V3 c, int axis) { return axis == 0 ? c.x : (axis == 1 ? c.y : c.z); }

struct BuildCfg {
    int heuristic;  // 0 Midpoint, 1 Sah
    uint32_t splits;
    int mode;  // 0 literal (O(splits*n) per node, exactly as coded), 1 fast (prefix/suffix
               // boxes + de-duplicated split indices; min/max are exact so the tree is identical)
};

// BvhData::sort bvh.rs:100-139 — Rust sort_by is a stable merge sort; objects and centres are
// sorted independently on the same keys.
static void sort_axis(std::vector<const Object*>& objs, std::vector<V3>& centers, int axis) {
    std::vector<size_t> idx(objs.size());
    for (size_t i = 0; i < idx.size(); ++i) idx[i] = i;
    std::stable_sort(idx.begin(), idx.end(), [&](size_t a, size_t b) {
        return axis_of(centers[a], axis) < axis_of(centers[b], axis);
    });
    std::vector<const Object*> o2(objs.size());
    std::vector<V3> c2(objs.size());
    for (size_t i = 0; i < idx.size(); ++i) {
        o2[i] = objs[idx[i]];
        c2[i] = centers[idx[i]];
    }
    objs.swap(o2);
    centers.swap(c2);
}

// split_ind bvh.rs:7-13: first k with centre_k > split, None if none.
static inline long split_ind_literal(const std::vector<V3>& centers, int axis, double split) {
    for (size_t k = 0; k < centers.size(); ++k)
        if (axis_of(centers[k], axis) > split) return (long)k;
    return -1;
}

// calculate_sah bvh.rs:15-38
static double calculate_sah_literal(double cost_traversal, double cost_intersect, double surface_area,
                                    const std::vector<const Object*>& objs, size_t ind) {
    double p_left = 0., p_right = 0.;
    size_t n = objs.size();
    if (ind > 0) p_left = bbox_of(objs, 0, ind).surface_area() / surface_area;
    if (ind < n) p_right = bbox_of(objs, ind, n).surface_area() / surface_area;
    return cost_traversal + cost_intersect * (p_left * (double)ind + p_right * (double)(n - ind));
}

static std::unique_ptr<BvhTree> build_tree(std::vector<const Object*> objs, std::vector<V3> centers,
                                           const BuildCfg& cfg) {
    // build_sah bvh.rs:227-317 / build_midpoint bvh.rs:319-389
    size_t n = objs.size();
    AABB bbox = bbox_of(objs, 0, n);
    auto node = std::make_unique<BvhTree>();
    node->leaf = false;
    node->box = bbox;
    node->obj = nullptr;
    if (n > 4) {
        double x = bbox.xmax - bbox.xmin, y = bbox.ymax - bbox.ymin, z = bbox.zmax - bbox.zmin;
        int axis;
        double amin, alen;
        if (x >= y && x >= z) { axis = 0; amin = bbox.xmin; alen = x; }
        else if (y >= z) { axis = 1; amin = bbox.ymin; alen = y; }
        else { axis = 2; amin = bbox.zmin; alen = z; }
        sort_axis(objs, centers, axis);
        long ind = -1;
        if (cfg.heuristic == 1) {
            double surface_area = bbox.surface_area();
            double split_dist = alen / (double)(cfg.splits - 1);
            double min_sah = std::numeric_limits<double>::infinity();
            if (cfg.mode == 0) {
                for (uint32_t i = 1; i < cfg.splits + 1; ++i) {
                    long k = split_ind_literal(centers, axis, amin + (double)i * split_dist);
                    if (k >= 0) {
                        double sah = calculate_sah_literal(0.3, 1., surface_area, objs, (size_t)k);
                        if (sah < min_sah) { min_sah = sah; ind = k; }
                    }
                }
            } else {
                // prefix/suffix boxes: left(k) = box of [0,k), right(k) = box of [k,n)
                std::vector<AABB> pre(n + 1), suf(n + 1);
                for (size_t k = 0; k < n; ++k) pre[k + 1] = (k == 0) ? objs[0]->bbox() : pre[k].expand(objs[k]->bbox());
                for (size_t k = n; k-- > 0;) suf[k] = (k == n - 1) ? objs[k]->bbox() : objs[k]->bbox().expand(suf[k + 1]);
                // NB expand() is min/max per component: exact and order independent, so
                // pre/suf equal the reference's left-to-right folds bit for bit.
                std::vector<double> keys(n);
                for (size_t k = 0; k < n; ++k) keys[k] = axis_of(centers[k], axis);
                long last = -2;
                for (uint32_t i = 1; i < cfg.splits + 1; ++i) {
                    double thr = amin + (double)i * split_dist;
                    size_t k = std::upper_bound(keys.begin(), keys.end(), thr) - keys.begin();
                    if (k >= n) continue;  // None
                    if ((long)k == last) continue;  // same index => same cost, strict < keeps the first
                    last = (long)k;
                    double p_left = k > 0 ? pre[k].surface_area() / surface_area : 0.;
                    double p_right = suf[k].surface_area() / surface_area;
                    double sah = 0.3 + 1. * (p_left * (double)k + p_right * (double)(n - k));
                    if (sah < min_sah) { min_sah = sah; ind = (long)k; }
                }
            }
        } else {
            double split = axis_of(bbox.center(), axis);
            ind = split_ind_literal(centers, axis, split);
        }
        if (ind < 0 || ind == 0 || ind == (long)n - 1) ind = (long)(n / 2);
        std::vector<const Object*> lo(objs.begin(), objs.begin() + ind), ro(objs.begin() + ind, objs.end());
        std::vector<V3> lc(centers.begin(), centers.begin() + ind), rc(centers.begin() + ind, centers.end());
        objs.clear(); objs.shrink_to_fit();
        centers.clear(); centers.shrink_to_fit();
        auto make_side = [&](std::vector<const Object*>& so, std::vector<V3>& sc) {
            if (so.size() > 1) return build_tree(std::move(so), std::move(sc), cfg);
            auto leaf = std::make_unique<BvhTree>();
            leaf->leaf = true;
            leaf->obj = so[0];
            return leaf;
        };
        node->children.push_back(make_side(lo, lc));
        node->children.push_back(make_side(ro, rc));
    } else {
        for (size_t i = 0; i < n; ++i) {
            auto leaf = std::make_unique<BvhTree>();
            leaf->leaf = true;
            leaf->obj = objs[i];
            node->children.push_back(std::move(leaf));
        }
    }
    return node;
}

// ------------------------------------------------------------------------------------
// Scene (lib.rs:216-296)
// ------------------------------------------------------------------------------------
struct Scene {
    std::vector<Object> objects;
    std::vector<Material> materials;
    std::vector<Emission> emissions;
    std::unique_ptr<BvhTree> bvh;
    double tmin, tmax;
    size_t hdri_w, hdri_h;
    std::vector<V3> hdri;

    V3 hdri_pixel(size_t i, size_t j) const {
        // Image::pixel image.rs:183-186 asserts i<height && j<width; at theta==pi or
        // phi==2pi exactly the reference would panic.  The oracle clamps (measure-zero case).
        if (i >= hdri_h) i = hdri_h - 1;
        if (j >= hdri_w) j = hdri_w - 1;
        return hdri[i * hdri_w + j];
    }
    // Scene::background lib.rs:254-285
    V3 background(V3 dir) const {
        dir = unit(dir);
        double phi = std::atan2(dir.z, dir.x) + PI;
        double theta = std::acos(dir.y);
        double x = phi / (2. * PI) * (double)(hdri_w - 1);
        double y = theta / PI * (double)(hdri_h - 1);
        double x_f = std::floor(x), x_c = std::ceil(x), y_f = std::floor(y), y_c = std::ceil(y);
        size_t i = (size_t)y_f, j = (size_t)x_f;
        V3 f0 = hdri_pixel(i, j), f1 = hdri_pixel(i + 1, j), f2 = hdri_pixel(i, j + 1), f3 = hdri_pixel(i + 1, j + 1);
        return f0 * (x_c - x) * (y_c - y) + f1 * (x_c - x) * (y - y_f) + f2 * (x - x_f) * (y_c - y) +
               f3 * (x - x_f) * (y - y_f);
    }
};

// Camera lib.rs:56-210 (derived fields only)
struct Camera {
    V3 origin, e_x, e_y, z;
    double width, height;
    uint32_t ppc;
};

static Camera camera_new(V3 origin, V3 up, V3 lookat, double fov, double width, double height, uint32_t ppi) {
    Camera c;
    c.ppc = (uint32_t)std::round((double)ppi * 2.54);  // lib.rs:113 (round half away from zero)
    V3 z = unit(lookat - origin);
    V3 x = unit(cross(up, z));
    V3 y = unit(cross(z, x));
    c.origin = origin;
    c.e_x = x;
    c.e_y = y;
    c.width = width;
    c.height = height;
    double rad = fov * (PI / 180.0);  // f64::to_radians
    c.z = (width / std::tan(rad / 2.)) * z;  // lib.rs:131
    return c;
}
static inline size_t camera_x_pixels(const Camera& c) { return (size_t)std::round(c.width * (double)c.ppc); }
static inline size_t camera_y_pixels(const Camera& c) { return (size_t)std::round(c.height * (double)c.ppc); }
// lib.rs:202-210
static inline Ray camera_primary_ray(const Camera& c, size_t i, size_t j, double r1, double r2) {
    double fi = (double)i, fj = (double)j;
    double x = (fj + r1) / (double)c.ppc - c.width / 2.;
    double y = (fi + r2) / (double)c.ppc - c.height / 2.;
    return Ray{c.origin, c.z + x * c.e_x + y * c.e_y};
}

// ------------------------------------------------------------------------------------
// Environment importance sampling (the GPU backend's RRS_FLAG_ENV_SAMPLING; not part of the reference).  Restates
// rayrs_b200/csrc/api.cu build_env_table / quantize_cdf (the table, bit for bit: the same f64 arithmetic, fp32
// arrays) and env.cuh (sampler, density, nee_bsdf, MIS weights) in f64.
// ------------------------------------------------------------------------------------
struct EnvTable {
    bool ok = true;                  // false: a non-finite texel (the render refuses the flag)
    uint32_t cw = 0, ch = 0;         // cells: hdri_w - 1, hdri_h - 1
    std::vector<float> marg, cond;   // CDF starts, multiples of 2^-24; marg empty: a black map
    std::vector<float> cos0, dcos;   // per row: cos theta at the top edge, cos top - cos bottom
    float inv_dphi = 0.f;            // cw / 2pi
};

static bool quantize_cdf(const double* w, size_t n, double sum, float* start) {
    const int64_t G = 1 << 24;
    std::vector<int64_t> k(n);
    int64_t tot = 0;
    size_t big = 0;
    for (size_t j = 0; j < n; ++j) {
        k[j] = w[j] > 0. ? std::max<int64_t>(1, std::llround(w[j] / sum * (double)G)) : 0;
        tot += k[j];
        if (k[j] > k[big]) big = j;
    }
    k[big] += G - tot;
    if (k[big] < 1) return false;
    int64_t acc = 0;
    for (size_t j = 0; j < n; ++j) {
        start[j] = std::ldexp((float)acc, -24);
        acc += k[j];
    }
    return true;
}

static void build_env_table(const std::vector<V3>& hdri, size_t w, size_t h, EnvTable& out) {
    out = EnvTable();
    const uint32_t cw = (uint32_t)w - 1, ch = (uint32_t)h - 1;
    out.cw = cw;
    out.ch = ch;
    out.inv_dphi = (float)(cw / (2. * PI));
    for (const V3& t : hdri)
        if (!std::isfinite((float)t.x) || !std::isfinite((float)t.y) || !std::isfinite((float)t.z)) {
            out.ok = false;
            return;
        }
    auto lum = [&](uint32_t i, uint32_t j) {
        const V3& t = hdri[(size_t)i * w + j];
        return std::max(std::fabs((float)t.x), std::max(std::fabs((float)t.y), std::fabs((float)t.z)));
    };
    std::vector<double> cell((size_t)cw * ch), rows(ch);
    out.cos0.resize(ch);
    out.dcos.resize(ch);
    const double dphi = 2. * PI / cw;
    double total = 0.;
    for (uint32_t i = 0; i < ch; ++i) {
        const double t0 = PI * i / ch, t1 = PI * (i + 1) / ch;
        const double dcos = 2. * std::sin(0.5 * (t0 + t1)) * std::sin(0.5 * (t1 - t0));
        out.cos0[i] = (float)std::cos(t0);
        out.dcos[i] = (float)dcos;
        double r = 0.;
        for (uint32_t j = 0; j < cw; ++j) {
            const float m = std::max(std::max(lum(i, j), lum(i, j + 1)), std::max(lum(i + 1, j), lum(i + 1, j + 1)));
            const double c = (double)m * dphi * dcos;
            cell[(size_t)i * cw + j] = c;
            r += c;
        }
        rows[i] = r;
        total += r;
    }
    if (!std::isfinite(total)) { out.ok = false; return; }
    if (total == 0.) return;
    out.marg.resize(ch);
    out.cond.assign((size_t)cw * ch, 0.f);
    bool ok = quantize_cdf(rows.data(), ch, total, out.marg.data());
    for (uint32_t i = 0; i < ch && ok; ++i)
        if (rows[i] > 0.) ok = quantize_cdf(cell.data() + (size_t)i * cw, cw, rows[i], out.cond.data() + (size_t)i * cw);
    if (!ok) {
        out.ok = false;
        out.marg.clear();
        out.cond.clear();
    }
}

// largest k < n with a[k] <= u; the step of cell k (exact: multiples of 2^-24)
static inline uint32_t cdf_find(const float* a, uint32_t n, double u) {
    return (uint32_t)(std::upper_bound(a + 1, a + n, u, [](double x, float y) { return x < (double)y; }) - a) - 1u;
}
static inline double cdf_step(const float* a, uint32_t n, uint32_t k) { return (k + 1u < n ? (double)a[k + 1u] : 1.) - (double)a[k]; }

static inline double env_cell_pdf(const EnvTable& e, uint32_t i, uint32_t j) {
    const double pm = cdf_step(e.marg.data(), e.ch, i), pc = cdf_step(e.cond.data() + (size_t)i * e.cw, e.cw, j);
    return pm * pc * (double)e.inv_dphi / (double)e.dcos[i];
}

// the cell Scene::background reads direction dir from
static inline void env_cell_of(const Scene& s, const EnvTable& e, V3 dir, uint32_t& i, uint32_t& j) {
    dir = unit(dir);
    const double x = (std::atan2(dir.z, dir.x) + PI) / (2. * PI) * (double)(s.hdri_w - 1);
    const double y = std::acos(std::fmin(1., std::fmax(-1., dir.y))) / PI * (double)(s.hdri_h - 1);
    j = std::min((uint32_t)std::floor(x), e.cw - 1u);
    i = std::min((uint32_t)std::floor(y), e.ch - 1u);
}

static inline double env_pdf(const Scene& s, const EnvTable& e, V3 dir) {
    if (e.marg.empty()) return 0.;
    uint32_t i, j;
    env_cell_of(s, e, dir, i, j);
    return env_cell_pdf(e, i, j);
}

// (hi0, hi1): multiples of 2^-24 that pick the row and the cell; hi + 2^-24 lo places the direction inside it.
// Returns the density of the drawn cell.
static inline double env_sample(const EnvTable& e, double hi0, double hi1, double lo0, double lo1, V3& dir, uint32_t& i,
                                uint32_t& j) {
    i = cdf_find(e.marg.data(), e.ch, hi0);
    const double pm = cdf_step(e.marg.data(), e.ch, i);
    const float* cond = e.cond.data() + (size_t)i * e.cw;
    j = cdf_find(cond, e.cw, hi1);
    const double pc = cdf_step(cond, e.cw, j);
    const double t0 = std::fmin(((hi0 - (double)e.marg[i]) + lo0 / 16777216.0) / pm, 1.);
    const double t1 = std::fmin(((hi1 - (double)cond[j]) + lo1 / 16777216.0) / pc, 1.);
    const double cy = (double)e.cos0[i] - t0 * (double)e.dcos[i];
    const double sy = std::sqrt(std::fmax(0., (1. - cy) * (1. + cy)));
    const double phi = 2. * PI * ((double)j + t1) / (double)e.cw;
    dir = v3(-sy * std::cos(phi), cy, -sy * std::sin(phi));
    return env_cell_pdf(e, i, j);
}

// a uniform in [0, 1) split as the device draws it: the 24-bit part that picks the cell and the rest (in [0, 1))
static inline void env_split(double u, double& hi, double& lo) {
    const double x = std::ldexp(std::fmin(std::fmax(u, 0.), 1.), 24);
    const double f = std::fmin(std::floor(x), 16777215.);
    hi = std::ldexp(f, -24);
    lo = std::fmin(x - f, 1.);
}

// env.cuh nee_bsdf: W = the plain estimator's weight for direction l, return = the density with which the plain
// render produces l (0: never).  Cook-Torrance: Beckmann D from tan^2 = |n x h|^2 / nh^2, 0 from tan^2 / alpha^2 >= 80
// on (the device's cut-off), half-vector density D cos theta_h mirrored (1 / (4 h.v)).
static inline double nee_bsdf(const Material& m, V3 n, V3 v, V3 l, V3& W) {
    W = v3(0., 0., 0.);
    if (m.tag == MAT_LAMBERTIAN) {
        const double nl = dot(n, l);
        if (!(nl > 0.)) return 0.;
        W = m.color;
        return nl * FRAC_1_PI;
    }
    const V3 hh = v + l;
    if (is_zeros(hh)) return 0.;
    const V3 h = unit(hh);
    const double nh = dot(n, h), hv = dot(h, v), nl = dot(n, l), nv = std::fabs(dot(n, v));
    if (!(nh > 0.) || !(hv > 0.) || nl <= 0. || nv == 0.) return 0.;
    const double g = rmin(2. * nh * nv / hv, rmin(2. * nh * nl / hv, 1.));
    const V3 F = fresnel_value(m, m.fresnel_kind, h, v, ENTERING);
    W = m.color * F * (g * dot(h, l) / nv);
    const V3 c = cross(n, h);
    const double t = dot(c, c) / (nh * nh * m.alpha2);
    if (!(t < 80.)) return 0.;
    const double nh2 = nh * nh;
    return std::exp(-t) / (PI * m.alpha2 * nh2 * nh2) * nh / (4. * hv);
}

// power heuristic a^2 / (a^2 + b^2) and the cross term a b / (a^2 + b^2), at least one of a, b positive
static inline double mis_power(double a, double b) {
    const double s = rmin(a, b) / rmax(a, b), s2 = s * s;
    return (a >= b ? 1. : s2) / (1. + s2);
}
static inline double mis_cross(double a, double b) {
    const double s = rmin(a, b) / rmax(a, b);
    return s / (1. + s * s);
}

struct PathStats {
    uint64_t rays = 0;        // Bvh::intersect calls (shadow rays included)
    uint64_t shadow_rays = 0; // of which environment shadow rays
    uint64_t scatters = 0;
    uint64_t nan_pixels = 0;
    uint64_t neg_pixels = 0;
    // diagnostics of the sphere re-entry quirk (SURVEY.md F7): rays spawned ON a sphere that point
    // into it, and how many of them lose the far-side hit because the near root came out >= 0
    uint64_t reentry_total = 0;
    uint64_t reentry_lost = 0;
};

// radiance lib.rs:521-560.  env != nullptr: with next-event estimation of the environment as the GPU backend's
// RRS_FLAG_ENV_SAMPLING does it (wavefront.cu shade_hit / env_miss): at a Lambertian vertex or a Cook-Torrance vertex
// with alpha^2 > 0 in fp32, below the last bounce, one direction from the table (RNG slot 0x100 + b) is traced as a
// shadow ray and adds throughput * W * background * min(p, 1) / p * mis_cross(p_e, p_b) if it escapes; the
// continuation's escape is weighted by mis_power(p_b, p_e) (1 where the shadow strategy cannot produce its direction).
static V3 radiance(const Scene& s, Ray r, uint32_t max_bounces, Rng& rng, PathStats& st, const EnvTable* env = nullptr) {
    V3 throughput = v3(1., 1., 1.);
    V3 light = v3(0., 0., 0.);
    const Object* origin_obj = nullptr;
    double wcont = 1.;  // MIS weight of the current ray's escape
    for (uint32_t b = 0; b < max_bounces; ++b) {
        st.rays++;
        Hit h = tree_intersect(s.bvh.get(), r, s.tmin, s.tmax);
        if (origin_obj) {  // diagnostics only (does not influence the result)
            const Sphere* sp = dynamic_cast<const Sphere*>(origin_obj->geom.get());
            if (sp && dot(r.d, r.o - sp->origin) < 0.) {
                double ts;
                st.reentry_total++;
                if (!(sp->intersect(r, ts) && ts > s.tmin)) st.reentry_lost++;
            }
        }
        if (h.hit) {
            origin_obj = h.obj;
            V3 position = r.point(h.t);
            V3 normal = h.obj->geom->normal(position);
            V3 view = unit(-1. * r.d);
            rng.load(b + 1);
            DrawSrc rs{rng.u, 0};
            const Material& mat = s.materials[h.obj->mat];
            ScatterEvent e = material_evaluate(mat, position, normal, view, rs);
            const bool nee = env && !env->marg.empty() && b + 1 < max_bounces &&
                             (mat.tag == MAT_LAMBERTIAN || (mat.tag == MAT_COOK_TORRANCE && (float)mat.alpha2 > 0.f));
            if (nee) {
                Rng re = rng;
                re.load(0x100u + b);
                double hi0 = re.u[0], hi1 = re.u[1], lo0 = re.u[2], lo1 = re.u[3];
                if (rng.mode != 1) { env_split(re.u[0], hi0, lo0); env_split(re.u[1], hi1, lo1); }
                V3 l, W;
                uint32_t ci, cj;
                const double pe = env_sample(*env, hi0, hi1, lo0, lo1, l, ci, cj);
                const double pb = pe > 0. ? nee_bsdf(mat, normal, view, l, W) : 0.;
                const V3 tw = throughput * W;
                const double p = rmax(rmax(tw.x, tw.y), tw.z);
                if (pb > 0. && p > 0.) {
                    const double k = rmin(p, 1.) / p * mis_cross(pe, pb);
                    st.rays++;
                    st.shadow_rays++;
                    if (!tree_intersect(s.bvh.get(), Ray{position, l}, s.tmin, s.tmax).hit)
                        light = light + tw * s.background(l) * k;
                }
            }
            if (e.scatter) {
                st.scatters++;
                V3 emit = h.obj->emission < 0 ? v3(0, 0, 0) : s.emissions[h.obj->emission].emit();
                light = light + throughput * emit;
                throughput = throughput * e.color;
                double p = rmax(rmax(throughput.x, throughput.y), throughput.z);
                if (rng.u[3] > p) return light;
                // DivAssign<f64> is a true per-component division vecmath.rs:708-714
                throughput.x /= p; throughput.y /= p; throughput.z /= p;
                r = e.ray;
                if (nee) {
                    V3 W;
                    const double pb = nee_bsdf(mat, normal, view, r.d, W);
                    const double pe = env_pdf(s, *env, r.d);
                    wcont = pe > 0. && pb > 0. ? mis_power(pb, pe) : 1.;
                } else {
                    wcont = 1.;
                }
            } else {
                return light;
            }
        } else {
            if (env) return light + throughput * wcont * s.background(r.d);
            return light + throughput * s.background(r.d);
        }
    }
    return light;
}

}  // namespace orc

// ======================================================================================
// C ABI (ctypes).  All arrays are caller-owned, row-major, doubles unless noted.
// ======================================================================================
using namespace orc;

struct OrcScene {
    Scene s;
    EnvTable env;  // the environment-sampling table of s's HDRI
    std::string err;
};

static Material material_from_row(const double* r) {
    Material m;
    m.tag = (int)r[0];
    m.color = v3(r[1], r[2], r[3]);
    m.alpha2 = r[4] * r[4];  // CookTorrance::new stores alpha*alpha material.rs:710-714
    m.ior = r[5];
    m.fresnel_kind = (int)r[6];
    m.r0 = v3(r[7], r[8], r[9]);
    m.spec = v3(r[7], r[8], r[9]);
    if (m.tag == MAT_CT_GLASS || m.tag == MAT_CT_REFRACT || m.tag == MAT_PLASTIC) m.fresnel_kind = FRESNEL_DIELECTRIC;
    return m;
}

extern "C" {

// objs: n_obj x 12  [type, mat, emission(-1 dark), payload x9]
//   sphere  (type 0): radius, ox, oy, oz
//   plane   (type 1): axis(0..5 = X,XRev,Y,YRev,Z,ZRev), umin, umax, vmin, vmax, pos
//   triangle(type 2): p1 xyz, p2 xyz, p3 xyz
// mats: n_mat x 12 (see Material); emis: n_emis x 4 [strength, r, g, b]
// hdri: hh x hw x 3
OrcScene* orc_scene_create(const double* objs, uint64_t n_obj, const double* mats, uint64_t n_mat,
                           const double* emis, uint64_t n_emis, int heuristic, uint32_t splits,
                           int build_mode, const double* hdri, uint64_t hw, uint64_t hh, double tmin,
                           double tmax) {
    auto* h = new OrcScene();
    Scene& s = h->s;
    s.tmin = tmin;
    s.tmax = tmax;
    s.objects.resize(n_obj);
    for (uint64_t i = 0; i < n_obj; ++i) {
        const double* r = objs + i * 12;
        Object& o = s.objects[i];
        o.mat = (int)r[1];
        o.emission = (int)r[2];
        o.id = (int)i;
        int type = (int)r[0];
        if (type == 0) o.geom.reset(new Sphere(r[3], v3(r[4], r[5], r[6])));
        else if (type == 1) o.geom.reset(new Plane((int)r[3], r[4], r[5], r[6], r[7], r[8]));
        else o.geom.reset(new Triangle(v3(r[3], r[4], r[5]), v3(r[6], r[7], r[8]), v3(r[9], r[10], r[11])));
    }
    for (uint64_t i = 0; i < n_mat; ++i) s.materials.push_back(material_from_row(mats + i * 12));
    for (uint64_t i = 0; i < n_emis; ++i)
        s.emissions.push_back(Emission{false, emis[i * 4], v3(emis[i * 4 + 1], emis[i * 4 + 2], emis[i * 4 + 3])});
    s.hdri_w = hw;
    s.hdri_h = hh;
    s.hdri.resize(hw * hh);
    for (uint64_t i = 0; i < hw * hh; ++i) s.hdri[i] = v3(hdri[i * 3], hdri[i * 3 + 1], hdri[i * 3 + 2]);
    build_env_table(s.hdri, hw, hh, h->env);
    // Bvh::build bvh.rs:199-210 -> BvhData::new :87-98
    std::vector<const Object*> ptrs(n_obj);
    std::vector<V3> centers(n_obj);
    for (uint64_t i = 0; i < n_obj; ++i) {
        ptrs[i] = &s.objects[i];
        centers[i] = s.objects[i].bbox().center();
    }
    BuildCfg cfg{heuristic, splits, build_mode};
    s.bvh = build_tree(std::move(ptrs), std::move(centers), cfg);
    return h;
}

void orc_scene_destroy(OrcScene* h) { delete h; }

// Pre-order dump of the tree: for every Node: [-(nchildren)] then its children; for every
// LeafNode: [object id].  boxes (optional) receives 6 doubles per Node in the same order.
// Returns the number of ints written (call with out=NULL to size).
static void dump_rec(const BvhTree* n, std::vector<int64_t>& out, std::vector<double>& boxes) {
    if (n->leaf) {
        out.push_back(n->obj->id);
        return;
    }
    out.push_back(-(int64_t)n->children.size());
    boxes.insert(boxes.end(), {n->box.xmin, n->box.xmax, n->box.ymin, n->box.ymax, n->box.zmin, n->box.zmax});
    for (const auto& c : n->children) dump_rec(c.get(), out, boxes);
}
uint64_t orc_tree_dump(const OrcScene* h, int64_t* out, uint64_t cap, double* boxes, uint64_t box_cap) {
    std::vector<int64_t> v;
    std::vector<double> b;
    dump_rec(h->s.bvh.get(), v, b);
    if (out) std::memcpy(out, v.data(), sizeof(int64_t) * std::min<uint64_t>(cap, v.size()));
    if (boxes) std::memcpy(boxes, b.data(), sizeof(double) * std::min<uint64_t>(box_cap, b.size()));
    return v.size();
}

// Closest hit for a batch of rays (rays: n x 6 = origin, direction).  obj_id = -1 on miss.
void orc_intersect(const OrcScene* h, const double* rays, uint64_t n, int32_t* obj_id, double* t, int nthreads) {
    const Scene& s = h->s;
    auto work = [&](uint64_t lo, uint64_t hi) {
        for (uint64_t i = lo; i < hi; ++i) {
            Ray r{v3(rays[i * 6], rays[i * 6 + 1], rays[i * 6 + 2]), v3(rays[i * 6 + 3], rays[i * 6 + 4], rays[i * 6 + 5])};
            Hit hit = tree_intersect(s.bvh.get(), r, s.tmin, s.tmax);
            obj_id[i] = hit.hit ? hit.obj->id : -1;
            t[i] = hit.hit ? hit.t : std::numeric_limits<double>::infinity();
        }
    };
    if (nthreads <= 1) { work(0, n); return; }
    std::vector<std::thread> th;
    uint64_t chunk = (n + nthreads - 1) / nthreads;
    for (int k = 0; k < nthreads; ++k) {
        uint64_t lo = std::min<uint64_t>(n, k * chunk), hi = std::min<uint64_t>(n, lo + chunk);
        th.emplace_back(work, lo, hi);
    }
    for (auto& x : th) x.join();
}

// Robustness of the closest-hit ID: a ray is "stable" iff the ID is unchanged under 12
// perturbations (direction +-eps*|d| and origin +-eps_o along each axis).  Rays that are not
// stable sit within ~eps of a decision boundary (primitive edge, silhouette, t-tie, box
// face) where an fp32 evaluation may legitimately decide differently.
//
// orc_intersect_sensitivity is the same probe with the largest relative change of t over the 12 perturbations
// written to `tchange` (0 for misses and for rays that are not stable): the conditioning of t with respect to
// the ray.  At grazing incidence on a triangle (|cos| ~ 0.01) a 2e-6 perturbation moves t by ~1e-4, and an
// fp32 evaluation, whose rounding acts like a perturbation of a few 1e-7, cannot be asked for 1e-5 there.
static void intersect_sensitivity(const OrcScene* h, const double* rays, uint64_t n, double eps_dir, double eps_org,
                                  uint8_t* stable, double* tchange, int nthreads) {
    const Scene& s = h->s;
    auto work = [&](uint64_t lo, uint64_t hi) {
        for (uint64_t i = lo; i < hi; ++i) {
            Ray r{v3(rays[i * 6], rays[i * 6 + 1], rays[i * 6 + 2]), v3(rays[i * 6 + 3], rays[i * 6 + 4], rays[i * 6 + 5])};
            Hit h0 = tree_intersect(s.bvh.get(), r, s.tmin, s.tmax);
            int id0 = h0.hit ? h0.obj->id : -1;
            double dl = mag(r.d) * eps_dir;
            bool ok = true;
            double worst = 0.0;
            for (int k = 0; k < 12 && ok; ++k) {
                Ray q = r;
                double sgn = (k & 1) ? -1. : 1.;
                int ax = (k >> 1) % 3;
                bool org = k >= 6;
                double* comp = org ? (ax == 0 ? &q.o.x : ax == 1 ? &q.o.y : &q.o.z)
                                   : (ax == 0 ? &q.d.x : ax == 1 ? &q.d.y : &q.d.z);
                *comp += sgn * (org ? eps_org : dl);
                Hit hk = tree_intersect(s.bvh.get(), q, s.tmin, s.tmax);
                int idk = hk.hit ? hk.obj->id : -1;
                if (idk != id0) ok = false;
                if (ok && hk.hit) {
                    double rel = std::fabs(hk.t - h0.t) / std::fabs(h0.t);
                    if (rel > 1e-3) ok = false;
                    worst = std::max(worst, rel);
                }
            }
            stable[i] = ok ? 1 : 0;
            if (tchange) tchange[i] = ok ? worst : 0.0;
        }
    };
    std::vector<std::thread> th;
    if (nthreads < 1) nthreads = 1;
    uint64_t chunk = (n + nthreads - 1) / nthreads;
    for (int k = 0; k < nthreads; ++k) {
        uint64_t lo = std::min<uint64_t>(n, k * chunk), hi = std::min<uint64_t>(n, lo + chunk);
        th.emplace_back(work, lo, hi);
    }
    for (auto& x : th) x.join();
}

void orc_intersect_stable(const OrcScene* h, const double* rays, uint64_t n, double eps_dir, double eps_org,
                          uint8_t* stable, int nthreads) {
    intersect_sensitivity(h, rays, n, eps_dir, eps_org, stable, nullptr, nthreads);
}

void orc_intersect_sensitivity(const OrcScene* h, const double* rays, uint64_t n, double eps_dir, double eps_org,
                               uint8_t* stable, double* tchange, int nthreads) {
    intersect_sensitivity(h, rays, n, eps_dir, eps_org, stable, tchange, nthreads);
}

// Camera::new -> derived fields.  out: origin(3) e_x(3) e_y(3) z(3) width height ppc xpix ypix
void orc_camera_new(const double* origin, const double* up, const double* lookat, double fov, double width,
                    double height, uint32_t ppi, double* out) {
    Camera c = camera_new(v3(origin[0], origin[1], origin[2]), v3(up[0], up[1], up[2]),
                          v3(lookat[0], lookat[1], lookat[2]), fov, width, height, ppi);
    double v[17] = {c.origin.x, c.origin.y, c.origin.z, c.e_x.x, c.e_x.y, c.e_x.z, c.e_y.x, c.e_y.y, c.e_y.z,
                    c.z.x, c.z.y, c.z.z, c.width, c.height, (double)c.ppc, (double)camera_x_pixels(c),
                    (double)camera_y_pixels(c)};
    std::memcpy(out, v, sizeof(v));
}

static Camera camera_from_derived(const double* d) {
    Camera c;
    c.origin = v3(d[0], d[1], d[2]);
    c.e_x = v3(d[3], d[4], d[5]);
    c.e_y = v3(d[6], d[7], d[8]);
    c.z = v3(d[9], d[10], d[11]);
    c.width = d[12];
    c.height = d[13];
    c.ppc = (uint32_t)d[14];
    return c;
}

// Primary rays exactly as the tile loop would generate them for image pixel (row, col) and
// global sample index s (F8 mapping main.rs:71-76).  out: n x 6.
void orc_primary_rays(const double* cam17, uint32_t W, uint32_t H, const uint32_t* rows, const uint32_t* cols,
                      const uint32_t* samples, uint64_t n, uint64_t seed, int rng_mode, double* out) {
    Camera c = camera_from_derived(cam17);
    for (uint64_t k = 0; k < n; ++k) {
        Rng rng{seed, rows[k] * W + cols[k], samples[k], rng_mode, {0, 0, 0, 0}};
        rng.load(0);
        Ray r = camera_primary_ray(c, (size_t)H - rows[k], (size_t)W - cols[k], rng.u[0], rng.u[1]);
        double v[6] = {r.o.x, r.o.y, r.o.z, r.d.x, r.d.y, r.d.z};
        std::memcpy(out + k * 6, v, sizeof(v));
    }
}

// The render call being replaced: rayrs/src/main.rs:52-94.  out: H x W x 3 mean radiance.
// stats_out: [rays, scatters, nan_pixels, negative_pixels, seconds*1e6, reentry_total, reentry_lost]
// env: with environment sampling (radiance); stats_out then has an 8th entry, the shadow rays (counted in rays too).
static void render(const OrcScene* h, const double* cam17, uint32_t W, uint32_t H, uint32_t spp, uint32_t sample_offset,
                   uint32_t max_bounces, uint64_t seed, int rng_mode, int nthreads, double* out, uint64_t* stats_out,
                   const EnvTable* env) {
    const Scene& s = h->s;
    Camera c = camera_from_derived(cam17);
    const uint32_t B = 16;  // main.rs:57
    uint32_t bx = (W + B - 1) / B, by = (H + B - 1) / B;
    std::atomic<uint32_t> next{0};
    if (nthreads < 1) nthreads = 1;
    std::vector<PathStats> stats(nthreads);
    auto t0 = std::chrono::steady_clock::now();
    auto work = [&](int tid) {
        PathStats& st = stats[tid];
        for (;;) {
            uint32_t b = next.fetch_add(1);
            if (b >= bx * by) break;
            uint32_t off_x = (b % bx) * B, off_y = (b / bx) * B;
            uint32_t bw = std::min(B, W - off_x), bh = std::min(B, H - off_y);
            for (uint32_t j = 0; j < bw; ++j) {
                for (uint32_t i = 0; i < bh; ++i) {
                    uint32_t row = i + off_y, col = j + off_x;
                    V3 pixel = v3(0., 0., 0.);
                    for (uint32_t k = 0; k < spp; ++k) {
                        Rng rng{seed, row * W + col, sample_offset + k, rng_mode, {0, 0, 0, 0}};
                        rng.load(0);
                        Ray r = camera_primary_ray(c, (size_t)H - i - off_y, (size_t)W - j - off_x, rng.u[0], rng.u[1]);
                        pixel = pixel + radiance(s, r, max_bounces, rng, st, env);
                    }
                    if (std::isnan(pixel.x) || std::isnan(pixel.y) || std::isnan(pixel.z)) st.nan_pixels++;
                    if (pixel.x < 0. || pixel.y < 0. || pixel.z < 0.) st.neg_pixels++;
                    V3 m = pixel / (double)spp;  // main.rs:89
                    double* o = out + ((uint64_t)row * W + col) * 3;
                    o[0] = m.x; o[1] = m.y; o[2] = m.z;
                }
            }
        }
    };
    std::vector<std::thread> th;
    for (int k = 0; k < nthreads; ++k) th.emplace_back(work, k);
    for (auto& x : th) x.join();
    auto t1 = std::chrono::steady_clock::now();
    if (stats_out) {
        PathStats tot;
        for (auto& st : stats) {
            tot.rays += st.rays; tot.scatters += st.scatters;
            tot.nan_pixels += st.nan_pixels; tot.neg_pixels += st.neg_pixels;
            tot.reentry_total += st.reentry_total; tot.reentry_lost += st.reentry_lost;
            tot.shadow_rays += st.shadow_rays;
        }
        stats_out[0] = tot.rays;
        stats_out[1] = tot.scatters;
        stats_out[2] = tot.nan_pixels;
        stats_out[3] = tot.neg_pixels;
        stats_out[4] = (uint64_t)std::chrono::duration_cast<std::chrono::microseconds>(t1 - t0).count();
        stats_out[5] = tot.reentry_total;
        stats_out[6] = tot.reentry_lost;
        if (env) stats_out[7] = tot.shadow_rays;
    }
}

void orc_render(const OrcScene* h, const double* cam17, uint32_t W, uint32_t H, uint32_t spp,
                uint32_t sample_offset, uint32_t max_bounces, uint64_t seed, int rng_mode, int nthreads,
                double* out, uint64_t* stats_out) {
    render(h, cam17, W, H, spp, sample_offset, max_bounces, seed, rng_mode, nthreads, out, stats_out, nullptr);
}

// orc_render with environment sampling (RRS_FLAG_ENV_SAMPLING).  stats_out: 8 entries, the last the shadow rays.
// Returns -1 (and renders nothing) if the map has a non-finite texel, as the GPU backend refuses the flag.
int orc_render_env(const OrcScene* h, const double* cam17, uint32_t W, uint32_t H, uint32_t spp, uint32_t sample_offset,
                   uint32_t max_bounces, uint64_t seed, int rng_mode, int nthreads, double* out, uint64_t* stats_out) {
    if (!h->env.ok) return -1;
    render(h, cam17, W, H, spp, sample_offset, max_bounces, seed, rng_mode, nthreads, out, stats_out, &h->env);
    return 0;
}

// The sampling table: returns 1 (tabulated), 0 (black map: empty table) or -1 (non-finite texels).  Each of marg
// (ch floats), cond (ch x cw floats) and row (ch x 2 floats: cos theta at the top edge, cos top - cos bottom) may be
// null; they are written only for a tabulated map.
int orc_env_table(const OrcScene* h, float* marg, float* cond, float* row) {
    const EnvTable& e = h->env;
    if (!e.ok) return -1;
    if (e.marg.empty()) return 0;
    if (marg) std::memcpy(marg, e.marg.data(), sizeof(float) * e.marg.size());
    if (cond) std::memcpy(cond, e.cond.data(), sizeof(float) * e.cond.size());
    if (row)
        for (uint32_t i = 0; i < e.ch; ++i) { row[2 * i] = e.cos0[i]; row[2 * i + 1] = e.dcos[i]; }
    return 1;
}

// rrs_env_sample's inputs: u n x 2 uniforms in [0, 1), each split into the 24 bits that pick the cell and the rest.
// out: n x 6 = direction xyz, density of the drawn cell, cell row, cell column.  -1 if the table is empty or refused.
int orc_env_sample(const OrcScene* h, const double* u, uint64_t n, double* out) {
    const EnvTable& e = h->env;
    if (!e.ok || e.marg.empty()) return -1;
    for (uint64_t k = 0; k < n; ++k) {
        double hi0, lo0, hi1, lo1;
        env_split(u[2 * k], hi0, lo0);
        env_split(u[2 * k + 1], hi1, lo1);
        V3 d;
        uint32_t i, j;
        const double pdf = env_sample(e, hi0, hi1, lo0, lo1, d, i, j);
        double v[6] = {d.x, d.y, d.z, pdf, (double)i, (double)j};
        std::memcpy(out + 6 * k, v, sizeof(v));
    }
    return 0;
}

// rrs_env_pdf: the density of n directions (n x 3) in the cell background() reads them from.  -1 if refused.
int orc_env_pdf(const OrcScene* h, const double* dirs, uint64_t n, double* pdf) {
    if (!h->env.ok) return -1;
    for (uint64_t k = 0; k < n; ++k) pdf[k] = env_pdf(h->s, h->env, v3(dirs[3 * k], dirs[3 * k + 1], dirs[3 * k + 2]));
    return 0;
}

// Material::evaluate for a batch.  mat_row: 12 doubles.  nv: n x 6 (normal, view — both unit).
// u: n x 3 material draws.  out: n x 7 [scatter flag, color rgb, direction xyz]
void orc_material_evaluate(const double* mat_row, const double* nv, const double* u, uint64_t n, double* out) {
    Material m = material_from_row(mat_row);
    for (uint64_t i = 0; i < n; ++i) {
        V3 nrm = v3(nv[i * 6], nv[i * 6 + 1], nv[i * 6 + 2]);
        V3 view = v3(nv[i * 6 + 3], nv[i * 6 + 4], nv[i * 6 + 5]);
        double uu[4] = {u[i * 3], u[i * 3 + 1], u[i * 3 + 2], 0.};
        DrawSrc rs{uu, 0};
        ScatterEvent e = material_evaluate(m, v3(0, 0, 0), nrm, view, rs);
        double* o = out + i * 7;
        o[0] = e.scatter ? 1. : 0.;
        o[1] = e.color.x; o[2] = e.color.y; o[3] = e.color.z;
        o[4] = e.ray.d.x; o[5] = e.ray.d.y; o[6] = e.ray.d.z;
    }
}

// Material::evaluate with pdf = Some(Pdf::Hittable(light)) for a batch (the dormant next-event-estimation hook).
// obj_row: 12 doubles as orc_scene_create takes them (the light's geometry).  pnv: n x 9 (position, unit normal, unit view).
// u: n x 4 draws in call order.  out: n x 7 as orc_material_evaluate.
void orc_material_evaluate_pdf(const double* mat_row, const double* obj_row, const double* pnv, const double* u, uint64_t n,
                               double* out) {
    Material m = material_from_row(mat_row);
    std::unique_ptr<Hittable> g;
    const double* r = obj_row;
    int type = (int)r[0];
    if (type == 0) g.reset(new Sphere(r[3], v3(r[4], r[5], r[6])));
    else if (type == 1) g.reset(new Plane((int)r[3], r[4], r[5], r[6], r[7], r[8]));
    else g.reset(new Triangle(v3(r[3], r[4], r[5]), v3(r[6], r[7], r[8]), v3(r[9], r[10], r[11])));
    for (uint64_t i = 0; i < n; ++i) {
        const double* q = pnv + i * 9;
        double uu[4] = {u[i * 4], u[i * 4 + 1], u[i * 4 + 2], u[i * 4 + 3]};
        DrawSrc rs{uu, 0};
        ScatterEvent e = material_evaluate(m, v3(q[0], q[1], q[2]), v3(q[3], q[4], q[5]), v3(q[6], q[7], q[8]), rs, g.get());
        double* o = out + i * 7;
        o[0] = e.scatter ? 1. : 0.;
        o[1] = e.color.x; o[2] = e.color.y; o[3] = e.color.z;
        o[4] = e.ray.d.x; o[5] = e.ray.d.y; o[6] = e.ray.d.z;
    }
}
// Hittable::area and one Hittable::sample of the same row (u2: the two draws) -> out4 = [area, point xyz]
void orc_hittable_area_sample(const double* obj_row, const double* u2, double* out4) {
    const double* r = obj_row;
    std::unique_ptr<Hittable> g;
    int type = (int)r[0];
    if (type == 0) g.reset(new Sphere(r[3], v3(r[4], r[5], r[6])));
    else if (type == 1) g.reset(new Plane((int)r[3], r[4], r[5], r[6], r[7], r[8]));
    else g.reset(new Triangle(v3(r[3], r[4], r[5]), v3(r[6], r[7], r[8]), v3(r[9], r[10], r[11])));
    double uu[2] = {u2[0], u2[1]};
    DrawSrc rs{uu, 0};
    V3 p = g->sample(rs);
    out4[0] = g->area(); out4[1] = p.x; out4[2] = p.y; out4[3] = p.z;
}

// Scene::background for a batch of directions (n x 3) -> n x 3
void orc_background(const OrcScene* h, const double* dirs, uint64_t n, double* out) {
    for (uint64_t i = 0; i < n; ++i) {
        V3 c = h->s.background(v3(dirs[i * 3], dirs[i * 3 + 1], dirs[i * 3 + 2]));
        out[i * 3] = c.x; out[i * 3 + 1] = c.y; out[i * 3 + 2] = c.z;
    }
}

// Primitive-level entry points for the reference's known-answer tests.
int orc_sphere_intersect(double radius, const double* origin, const double* ray6, double* t) {
    Sphere s(radius, v3(origin[0], origin[1], origin[2]));
    Ray r{v3(ray6[0], ray6[1], ray6[2]), v3(ray6[3], ray6[4], ray6[5])};
    return s.intersect(r, *t) ? 1 : 0;
}
int orc_plane_intersect(int axis, double umin, double umax, double vmin, double vmax, double pos,
                        const double* ray6, double* t) {
    Plane p(axis, umin, umax, vmin, vmax, pos);
    Ray r{v3(ray6[0], ray6[1], ray6[2]), v3(ray6[3], ray6[4], ray6[5])};
    return p.intersect(r, *t) ? 1 : 0;
}
int orc_triangle_intersect(const double* p9, const double* ray6, double* t, double* normal3) {
    Triangle tr(v3(p9[0], p9[1], p9[2]), v3(p9[3], p9[4], p9[5]), v3(p9[6], p9[7], p9[8]));
    Ray r{v3(ray6[0], ray6[1], ray6[2]), v3(ray6[3], ray6[4], ray6[5])};
    if (normal3) { normal3[0] = tr.n.x; normal3[1] = tr.n.y; normal3[2] = tr.n.z; }
    return tr.intersect(r, *t) ? 1 : 0;
}
int orc_aabb_intersect(const double* box6, const double* ray6, double tmin, double tmax) {
    AABB b{box6[0], box6[1], box6[2], box6[3], box6[4], box6[5]};
    Ray r{v3(ray6[0], ray6[1], ray6[2]), v3(ray6[3], ray6[4], ray6[5])};
    return b.intersect(r, tmin, tmax) ? 1 : 0;
}
// bbox of the whole object list + derived quantities: out = box6, center3, volume, surface
void orc_scene_bbox(const OrcScene* h, double* out11) {
    const Scene& s = h->s;
    AABB b = s.objects[0].bbox();
    for (size_t i = 1; i < s.objects.size(); ++i) b = b.expand(s.objects[i].bbox());
    V3 c = b.center();
    double v[11] = {b.xmin, b.xmax, b.ymin, b.ymax, b.zmin, b.zmax, c.x, c.y, c.z, b.volume(), b.surface_area()};
    std::memcpy(out11, v, sizeof(v));
}
// The Vec3 operators as the restatement uses them, for the reference's own unit tests (vecmath.rs:816-881):
// out = [a + b, a - b, a * b, s * a, a * s, a . b, a x b, |a|^2] = 3 + 3 + 3 + 3 + 3 + 1 + 3 + 1 doubles
void orc_vecmath_ops(const double* a3, const double* b3, double s, double* out20) {
    V3 a = v3(a3[0], a3[1], a3[2]), b = v3(b3[0], b3[1], b3[2]);
    V3 r[5] = {a + b, a - b, a * b, s * a, a * s};
    for (int k = 0; k < 5; ++k) { out20[3 * k] = r[k].x; out20[3 * k + 1] = r[k].y; out20[3 * k + 2] = r[k].z; }
    out20[15] = dot(a, b);
    V3 c = cross(a, b);
    out20[16] = c.x; out20[17] = c.y; out20[18] = c.z;
    out20[19] = mag2(a);
}
void orc_orthonormal_basis(const double* n3, double* e1e2) {
    V3 e1, e2;
    orthonormal_basis(v3(n3[0], n3[1], n3[2]), e1, e2);
    double v[6] = {e1.x, e1.y, e1.z, e2.x, e2.y, e2.z};
    std::memcpy(e1e2, v, sizeof(v));
}
void orc_philox(const uint32_t* ctr4, const uint32_t* key2, uint32_t* out4, int rounds) {
    philox4x32(ctr4[0], ctr4[1], ctr4[2], ctr4[3], key2[0], key2[1], out4, rounds > 0 ? rounds : kPhiloxRounds);
}
// the uniforms of one RNG slot (4 doubles)
void orc_rng_uniforms(uint64_t seed, uint32_t pixel, uint32_t sample, uint32_t slot, int mode, double* out4) {
    Rng rng{seed, pixel, sample, mode, {0, 0, 0, 0}};
    rng.load(slot);
    std::memcpy(out4, rng.u, sizeof(double) * 4);
}

// Front-to-back, t-pruned traversal counts over the same tree, as a B200 stack traversal
// would do it (SURVEY.md 8(d)): for each ray, the number of child boxes tested and of
// primitives tested.  This defines N_nodes / N_prims in the bytes-per-ray model.
static void pruned_counts_rec(const BvhTree* n, const Ray& ray, double tmin, double& tbest, uint64_t& boxes,
                              uint64_t* prims) {
    // n is a Node whose own box has already been accepted
    struct Ent { const BvhTree* c; double entry; bool go; };
    Ent e[4];
    size_t k = n->children.size();
    for (size_t i = 0; i < k; ++i) {
        const BvhTree* c = n->children[i].get();
        e[i].c = c;
        if (c->leaf) {
            e[i].entry = 0.;
            e[i].go = true;
        } else {
            boxes++;
            e[i].go = c->box.intersect(ray, tmin, tbest);
            // entry distance for ordering
            double t0 = tmin;
            auto slab = [&](double lo, double hi, double o, double d) {
                double inv = 1. / d;
                double a = (lo - o) * inv, b = (hi - o) * inv;
                t0 = rmax(t0, rmin(a, b));
            };
            slab(c->box.xmin, c->box.xmax, ray.o.x, ray.d.x);
            slab(c->box.ymin, c->box.ymax, ray.o.y, ray.d.y);
            slab(c->box.zmin, c->box.zmax, ray.o.z, ray.d.z);
            e[i].entry = t0;
        }
    }
    if (k == 2 && !e[0].c->leaf && !e[1].c->leaf && e[1].entry < e[0].entry) std::swap(e[0], e[1]);
    for (size_t i = 0; i < k; ++i) {
        if (!e[i].go) continue;
        if (e[i].c->leaf) {
            const Hittable* g = e[i].c->obj->geom.get();
            prims[dynamic_cast<const Sphere*>(g) ? 0 : (dynamic_cast<const Plane*>(g) ? 1 : 2)]++;
            double t;
            if (g->intersect(ray, t) && t > tmin && t < tbest) tbest = t;
        } else {
            if (e[i].entry > tbest) continue;
            pruned_counts_rec(e[i].c, ray, tmin, tbest, boxes, prims);
        }
    }
}
// prims_out: 3 counters = spheres, planes, triangles tested
void orc_traversal_counts(const OrcScene* h, const double* rays, uint64_t n, uint64_t* boxes_out, uint64_t* prims_out,
                          uint64_t* hits_out) {
    const Scene& s = h->s;
    uint64_t boxes = 0, prims[3] = {0, 0, 0}, hits = 0;
    for (uint64_t i = 0; i < n; ++i) {
        Ray r{v3(rays[i * 6], rays[i * 6 + 1], rays[i * 6 + 2]), v3(rays[i * 6 + 3], rays[i * 6 + 4], rays[i * 6 + 5])};
        double tbest = s.tmax;
        boxes++;
        if (s.bvh->box.intersect(r, s.tmin, s.tmax)) pruned_counts_rec(s.bvh.get(), r, s.tmin, tbest, boxes, prims);
        if (tbest < s.tmax) hits++;
    }
    *boxes_out = boxes;
    prims_out[0] = prims[0]; prims_out[1] = prims[1]; prims_out[2] = prims[2];
    *hits_out = hits;
}

// Record the rays a render would trace (for bytes/ray statistics): the first `cap` rays of
// a single-threaded walk over pixels [0, npix) x samples [0, spp).
uint64_t orc_collect_path_rays(const OrcScene* h, const double* cam17, uint32_t W, uint32_t H, uint32_t spp,
                               uint32_t max_bounces, uint64_t seed, int rng_mode, uint32_t pixel_stride,
                               double* out_rays, uint64_t cap) {
    const Scene& s = h->s;
    Camera c = camera_from_derived(cam17);
    uint64_t cnt = 0;
    for (uint32_t pix = 0; pix < W * H && cnt < cap; pix += pixel_stride) {
        uint32_t row = pix / W, col = pix % W;
        for (uint32_t k = 0; k < spp && cnt < cap; ++k) {
            Rng rng{seed, pix, k, rng_mode, {0, 0, 0, 0}};
            rng.load(0);
            Ray r = camera_primary_ray(c, (size_t)H - row, (size_t)W - col, rng.u[0], rng.u[1]);
            V3 throughput = v3(1, 1, 1);
            for (uint32_t b = 0; b < max_bounces && cnt < cap; ++b) {
                double v[6] = {r.o.x, r.o.y, r.o.z, r.d.x, r.d.y, r.d.z};
                std::memcpy(out_rays + cnt * 6, v, sizeof(v));
                cnt++;
                Hit hit = tree_intersect(s.bvh.get(), r, s.tmin, s.tmax);
                if (!hit.hit) break;
                V3 position = r.point(hit.t);
                V3 normal = hit.obj->geom->normal(position);
                V3 view = unit(-1. * r.d);
                rng.load(b + 1);
                DrawSrc rs{rng.u, 0};
                ScatterEvent e = material_evaluate(s.materials[hit.obj->mat], position, normal, view, rs);
                if (!e.scatter) break;
                throughput = throughput * e.color;
                double p = rmax(rmax(throughput.x, throughput.y), throughput.z);
                if (rng.u[3] > p) break;
                throughput.x /= p; throughput.y /= p; throughput.z /= p;
                r = e.ray;
            }
        }
    }
    return cnt;
}

int orc_hardware_threads() { return (int)std::thread::hardware_concurrency(); }

}  // extern "C"
