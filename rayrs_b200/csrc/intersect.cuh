// fp32 primitive tests and the ordered, t-pruned stack traversal of the flattened reference
// BVH (production path).  Semantics follow rayrs-lib:
//   Sphere::intersect   geometry.rs:106-132     Plane::intersect  geometry.rs:229-271
//   Triangle::intersect geometry.rs:359-375     leaf filter t>tmin && t<tmax  bvh.rs:404-413
//   closest hit = smallest t, ties -> first leaf in DFS order (bvh.rs:50-72,395-399)
#pragma once
#include <cuda_fp16.h>

#include "device_types.cuh"

namespace rrs {

// 256-bit read-only loads (LDG.E.ENL2.256.CONSTANT on sm_100a): one instruction per node / primitive half.
// RRS_NODE_LD_HINT / RRS_PRIM_LD_HINT: L1 eviction priority of the node / primitive fetches (measurement switches:
// ".L1::evict_last", ".L1::evict_first", ".L1::no_allocate"; empty = evict_normal).
#ifndef RRS_NODE_LD_HINT
#define RRS_NODE_LD_HINT ""
#endif
#ifndef RRS_PRIM_LD_HINT
#define RRS_PRIM_LD_HINT ""
#endif
__device__ __forceinline__ void ldg256(const void* p, uint32_t (&v)[8]) {
    asm volatile("ld.global.nc" RRS_NODE_LD_HINT ".v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
                 : "l"(p));
}
__device__ __forceinline__ void ldg256(const void* p, float4& a, float4& b) {
    asm volatile("ld.global.nc" RRS_PRIM_LD_HINT ".v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=f"(a.x), "=f"(a.y), "=f"(a.z), "=f"(a.w), "=f"(b.x), "=f"(b.y), "=f"(b.z), "=f"(b.w)
                 : "l"(p));
}

__device__ __forceinline__ uint32_t prim_type(float4 a) { return __float_as_uint(a.w) & 3u; }
__device__ __forceinline__ uint32_t prim_material(float4 a) { return __float_as_uint(a.w) >> 2; }

// Sphere, cancellation-safe form (Haines et al., "Precision improvements for ray/sphere
// intersection").  Same decisions as the reference: needs desc > 0, returns the near root if
// it is >= 0, else the far root if that is >= 0.
//
// self == true: the ray was spawned ON this sphere.  In the f64 reference the near root is
// then +-1e-16 and its SIGN (rounding noise of the hit position) decides the outcome: near
// root >= 0 is returned and rejected by the leaf's t > tmin, so the far hit is lost; < 0
// falls through to the far root (SURVEY.md F7).  fp32 cannot reproduce that ray by ray;
// it reproduces it in distribution with the same mechanism: the sign of c = |o-centre|^2 - r^2
// evaluated on the fp32 hit position.
__device__ __forceinline__ bool hit_sphere(float4 a, float4 b, float3 o, float3 d, bool self, float& t) {
    float3 f = sub3(o, xyz(a));
    float r2 = b.x;
    float aa = dot3(d, d);
    float bp = -dot3(f, d);
    float c = dot3(f, f) - r2;
    if (self) {
        if (bp <= 0.f) return false;  // leaving the surface: both roots <= ~0 -> rejected by tmin
        if (c >= 0.f) return false;   // near root >= 0 -> returned -> rejected by tmin (F7)
    }
    float inv_a = 1.0f / aa;
    float3 l = madd3(d, bp * inv_a, f);  // f + (b'/a) d : closest approach to the centre
    float disc = r2 - dot3(l, l);        // == (b'^2 - a c) / a, without the cancellation
    if (!(disc > 0.f)) return false;
    float sq = sqrtf(aa * disc);
    float q = bp + copysignf(sq, bp);
    float t_a = q * inv_a;  // root of larger magnitude
    float t_b = c / q;      // the other root
    float t1 = fminf(t_a, t_b), t2 = fmaxf(t_a, t_b);
    if (self) {
        t = t2;
        return true;
    }
    if (t1 < 0.f) {
        if (t2 < 0.f) return false;
        t = t2;
        return true;
    }
    t = t1;
    return true;
}

// ---------------------------------------------------------------------------------------
// Sphere re-entry in f64.  A ray spawned ON a sphere and pointing into it (refraction) meets the
// reference's Sphere::intersect with a near root of ~+-1e-16; `t1 < 0` decides between "far root"
// and "near root returned, then rejected by the leaf's t > tmin" — i.e. the ray passes straight
// through the far side (SURVEY.md F7).  The sign of that near root is NOT noise: it is dominated by
// the f64 rounding of constants such as |camera - centre|^2 - r^2 in the intersection that produced
// the hit point, so the loss probability is a fixed property of the scene (measured in the oracle:
// 36 % for the sphere at x = 2.2, 81 % at x = +-6.6, 55 % at x = 0 of the seven-sphere scenes) and
// shows in the converged image.  No fp32 rule reproduces it.  Spheres with a transmissive material
// therefore get the reference's own arithmetic: hit distance, hit point and the re-entry test are
// evaluated in f64, operation for operation (no FMA contraction), and the f64 hit point travels
// with the ray.  Everything else stays fp32.
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ double dot64(double ax, double ay, double az, double bx, double by, double bz) {
    return __dadd_rn(__dadd_rn(__dmul_rn(ax, bx), __dmul_rn(ay, by)), __dmul_rn(az, bz));  // vecmath.rs:533-535
}
// Sphere::intersect geometry.rs:106-132, literally
__device__ __forceinline__ bool sphere_intersect64(double4 s, double ox, double oy, double oz, double dx, double dy,
                                                   double dz, double& t) {
    double odx = __dsub_rn(ox, s.x), ody = __dsub_rn(oy, s.y), odz = __dsub_rn(oz, s.z);
    double a = dot64(dx, dy, dz, dx, dy, dz);
    double b = __dmul_rn(2., dot64(dx, dy, dz, odx, ody, odz));
    double c = __dsub_rn(dot64(odx, ody, odz, odx, ody, odz), s.w);
    double desc = __dsub_rn(__dmul_rn(b, b), __dmul_rn(__dmul_rn(4., a), c));
    if (!(desc > 0.)) return false;
    double sq = __dsqrt_rn(desc);
    double t1 = __ddiv_rn(__dsub_rn(-b, sq), __dmul_rn(2., a));
    if (t1 < 0.) {
        double t2 = __ddiv_rn(__dadd_rn(-b, sq), __dmul_rn(2., a));  // only divided when it is needed
        if (t2 < 0.) return false;
        t = t2;
        return true;
    }
    t = t1;
    return true;
}

__device__ __forceinline__ bool sphere_reentry64(const DScene& sc, uint32_t sphere_index, const double* org64, float3 d, float* t) {
    double t64;
    const double4 s64 = sc.sphere64[sphere_index];
    const bool hit = sphere_intersect64(s64, org64[0], org64[1], org64[2], (double)d.x, (double)d.y, (double)d.z, t64) &&
                     t64 > sc.tmin64 && t64 < sc.tmax64;
    *t = (float)t64;
    return hit;
}

// Plane: a = (pos, umin, umax, meta), b = (vmin, vmax, axis, obj).  Half-open ranges, any
// sign of t is returned (the leaf filter removes t <= tmin).
__device__ __forceinline__ bool hit_plane(float4 a, float4 b, float3 o, float3 d, float& t) {
    uint32_t axis = __float_as_uint(b.z) >> 1;  // 0:x 1:y 2:z
    float ok = axis == 0 ? o.x : (axis == 1 ? o.y : o.z);
    float dk = axis == 0 ? d.x : (axis == 1 ? d.y : d.z);
    if (dk == 0.f) return false;
    float tt = (a.x - ok) / dk;
    float3 p = madd3(d, tt, o);
    float u = axis == 0 ? p.y : p.x;
    float v = axis == 2 ? p.y : p.z;
    if (u >= a.y && u < a.z && v >= b.x && v < b.y) {
        t = tt;
        return true;
    }
    return false;
}

// Triangle.  The reference is Moeller-Trumbore in f64 (geometry.rs:359-375): two-sided, edges
// inclusive (u >= 0, v >= 0, u + v <= 1), no determinant epsilon.  In fp32 that formulation leaks:
// with the origin ~10 units from a 0.007-unit triangle the barycentrics carry ~1e-4 of rounding
// and a ray can miss BOTH triangles of a shared edge (measured: ~1e-4 of rays on the 1M-triangle
// mesh passed through the surface).  The production test is therefore the watertight edge-function
// test of Woop, Benthin & Wald (JCGT 2013): vertices are translated to the ray origin and sheared
// into ray space; the edge function of a shared edge is computed from the SAME two projected
// vertices with exactly negated rounding in both triangles (no FMA contraction), so one of them
// always accepts.  Same decisions as the reference away from edges, same inclusive edges, two-sided.
//
// The shear is applied as two dot products with per-ray rows P = e_kx - Sx e_kz, Q = e_ky - Sy e_kz
// (entries 1, 0 and -S in ray-dependent positions) instead of per-vertex component selects: the
// projected coordinates of a vertex still depend on that vertex and the ray only — which is all
// watertightness needs — and the work moves from the ALU pipe (18 selects per triangle, the pipe
// that limits traversal: profiles/r01c_c4_fused_metrics.csv) to the half-idle FMA pipe.
struct RayProj {
    float3 P, Q;
};
__device__ __forceinline__ RayProj make_proj(float3 d) {
    // kz = the dominant axis of d, (kx, ky) = the next two axes cyclically, swapped when d[kz] < 0 (winding);
    // P = e_kx - (d[kx] / d[kz]) e_kz, Q = e_ky - (d[ky] / d[kz]) e_kz.  Written as one short arm per dominant axis
    // (a dozen instructions each, a warp takes at most three) instead of per-component selects (95 instructions).
    const float ax = fabsf(d.x), ay = fabsf(d.y), az = fabsf(d.z);
    RayProj r;
    if (ax > ay && ax > az) {         // kz = 0: (kx, ky) = (1, 2)
        const float sz = 1.0f / d.x, a = -d.y * sz, b = -d.z * sz;
        const float3 u = f3(a, 1.f, 0.f), v = f3(b, 0.f, 1.f);
        r.P = d.x < 0.f ? v : u;
        r.Q = d.x < 0.f ? u : v;
    } else if (!(ax > ay) && ay > az) {  // kz = 1: (kx, ky) = (2, 0)
        const float sz = 1.0f / d.y, a = -d.z * sz, b = -d.x * sz;
        const float3 u = f3(0.f, a, 1.f), v = f3(1.f, b, 0.f);
        r.P = d.y < 0.f ? v : u;
        r.Q = d.y < 0.f ? u : v;
    } else {                          // kz = 2: (kx, ky) = (0, 1)
        const float sz = 1.0f / d.z, a = -d.x * sz, b = -d.y * sz;
        const float3 u = f3(1.f, 0.f, a), v = f3(0.f, 1.f, b);
        r.P = d.z < 0.f ? v : u;
        r.Q = d.z < 0.f ? u : v;
    }
    return r;
}
__device__ __forceinline__ float proj3(float3 p, float3 v) {  // fixed association: part of the watertightness argument
    return __fmaf_rn(p.x, v.x, __fmaf_rn(p.y, v.y, __fmul_rn(p.z, v.z)));
}
__device__ __forceinline__ bool hit_triangle(float4 a, float4 b, float4 c, float3 o, float3 d, const RayProj& rp, float& t) {
    float3 A = sub3(xyz(a), o), B = sub3(xyz(b), o), C = sub3(xyz(c), o);
    float Ax = proj3(rp.P, A), Ay = proj3(rp.Q, A);
    float Bx = proj3(rp.P, B), By = proj3(rp.Q, B);
    float Cx = proj3(rp.P, C), Cy = proj3(rp.Q, C);
    float U = __fsub_rn(__fmul_rn(Cx, By), __fmul_rn(Cy, Bx));
    float V = __fsub_rn(__fmul_rn(Ax, Cy), __fmul_rn(Ay, Cx));
    float W = __fsub_rn(__fmul_rn(Bx, Ay), __fmul_rn(By, Ax));
    if (U == 0.f || V == 0.f || W == 0.f) {  // exactly on an edge in fp32: decide in fp64
        U = (float)((double)Cx * (double)By - (double)Cy * (double)Bx);
        V = (float)((double)Ax * (double)Cy - (double)Ay * (double)Cx);
        W = (float)((double)Bx * (double)Ay - (double)By * (double)Ax);
    }
    if (fminf(fminf(U, V), W) < 0.f && fmaxf(fmaxf(U, V), W) > 0.f) return false;
    float det = U + V + W;
    if (det == 0.f) return false;
    // hit point = barycentric mix of the translated vertices; its ray parameter is its projection on d
    float T = U * dot3(A, d) + V * dot3(B, d) + W * dot3(C, d);
    t = T / (det * dot3(d, d));
    return true;
}

// Hit distance of an ACCEPTED triangle hit, re-evaluated in f64 (Moeller-Trumbore as geometry.rs:359-375 writes it:
// t = (q . e2) / (p . e1), p = d x e2, q = (o - p1) x e1).  The fp32 projection test above decides WHETHER a triangle
// is hit (watertight) and which hit is closest; its distance carries three fp32 ulps of backward error, which at
// grazing incidence — where t itself is ill-conditioned — reached 1.28e-5 relative on one ray in 10^7
// (profiles/r01p_parity_measured.txt).  The closest hit's distance is therefore recomputed once per ray from the
// vertices the reference holds: the fp32 records when every vertex of the scene is exactly representable in fp32
// (PLY meshes), the f64 copy `tri64` otherwise.  ~45 f64 instructions per hit, outside the traversal loop.
__device__ __forceinline__ float triangle_t64(const DScene& sc, uint32_t pi, float4 a, float4 b, float4 c, float3 o, float3 d,
                                              float t32) {
    double p1x = a.x, p1y = a.y, p1z = a.z, p2x = b.x, p2y = b.y, p2z = b.z, p3x = c.x, p3y = c.y, p3z = c.z;
    if (sc.tri64 != nullptr) {
        const double* v = sc.tri64 + 9 * (size_t)pi;
        p1x = v[0]; p1y = v[1]; p1z = v[2]; p2x = v[3]; p2y = v[4]; p2z = v[5]; p3x = v[6]; p3y = v[7]; p3z = v[8];
    }
    const double e1x = p2x - p1x, e1y = p2y - p1y, e1z = p2z - p1z;
    const double e2x = p3x - p1x, e2y = p3y - p1y, e2z = p3z - p1z;
    const double tx = (double)o.x - p1x, ty = (double)o.y - p1y, tz = (double)o.z - p1z;
    const double dx = d.x, dy = d.y, dz = d.z;
    const double px = dy * e2z - dz * e2y, py = dz * e2x - dx * e2z, pz = dx * e2y - dy * e2x;
    const double qx = ty * e1z - tz * e1y, qy = tz * e1x - tx * e1z, qz = tx * e1y - ty * e1x;
    const double den = px * e1x + py * e1y + pz * e1z;
    const double t64 = (qx * e2x + qy * e2y + qz * e2z) / den;
    // a degenerate denominator (den ~ 0 in f64 while the fp32 projection accepted) keeps the fp32 value
    return fabs(t64 - (double)t32) <= 1e-2 * fabs((double)t32) ? (float)t64 : t32;
}

struct TravCounters {
    uint32_t nodes, prims;
};

// ---------------------------------------------------------------------------------------
// Ordered, t-pruned stack traversal, split into steps so that a warp can batch them
// (phase_extend in wavefront.cu keeps the 32 lanes on the same kind of step and refills idle lanes
// with new rays).  The per-thread stack is a column of a [entries][blockDim.x] shared-memory array
// (stride = blockDim.x -> conflict-free); entry 0 holds a TRAV_DONE sentinel so a pop needs no
// emptiness test.  TRAV_DONE == RRS_REF_EMPTY has the leaf bit set: "is an inner node" is one
// signed compare.
// ---------------------------------------------------------------------------------------
#define TRAV_DONE 0xFFFFFFFFu

// Per-thread traversal stack in shared memory, addressed by a 32-bit shared address held in a register: entry e
// of this thread lives at base + e * stride.  (As a generic pointer derived from threadIdx the compiler re-formed
// the address — S2R tid, S2UR cta-in-cluster, 4 more — inside every divergent push and pop: 4 % of the warp
// instructions of the traversal, profiles/r01n_c4.)
// Per-thread traversal stack in shared memory, addressed by a 32-bit shared address held in a register: entry e
// of this thread lives at base + e * stride.  (As a generic pointer derived from threadIdx the compiler re-formed
// the address — S2R tid, S2UR cta-in-cluster, 4 more — inside every divergent push and pop: 4 % of the warp
// instructions of the traversal, profiles/r01n_c4.)
// Measured alternatives (round 2, profiles/ab_logs/ab_r02c_stack.log, ab_r02f_hybrid.log): the whole stack in local
// memory (no shared memory, the SM's 256 KB almost all L1) -1.5 %; 15 entries in shared memory + local overflow
// -3.4 % / -1.6 % (the bound check in every push / pop costs more than the extra 35 KB of L1 brings).
struct SStack {
    uint32_t base;    // shared-window address of entry 0
    uint32_t stride;  // bytes between entries: 4 * threads per block
    __device__ __forceinline__ void init(const uint32_t* entry0, uint32_t threads) {
        uint32_t a = (uint32_t)__cvta_generic_to_shared(entry0);
        asm volatile("mov.u32 %0, %1;" : "=r"(base) : "r"(a));  // opaque: keep it, do not rematerialise it
        stride = 4u * threads;
    }
    __device__ __forceinline__ void set(uint32_t e, uint32_t v) const {
        asm volatile("st.shared.u32 [%0], %1;" ::"r"(base + e * stride), "r"(v));
    }
    __device__ __forceinline__ uint32_t get(uint32_t e) const {
        uint32_t v;
        asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(base + e * stride));
        return v;
    }
};

// The ray as the traversal keeps it in registers.
// Measured alternatives (round 2): (1) slab distances as one FMA per plane, t = plane * (1/d) - o * (1/d), with a
// PER-AXIS slack 2^-21 |o/d| folded into the near / far constants (round 1 had lost 36 % with one slack for all axes):
// 12 instructions fewer per node step, the same 28.64 node visits per ray — and 5 % SLOWER: the six extra per-ray
// constants doubled the kernel's spill traffic (local loads 326 M -> 635 M per launch), the L1 hit rate of the node
// fetches fell from 45.9 % to 43.2 % and issue-active from 70 % to 63 % (profiles/ab_logs/ncu_light_r02e_*.csv).
// (2) origin / direction / origin word parked in shared memory behind the stack and fetched back per leaf visit
// (9 registers fewer in the node loop): -15 % (ab_r02b_fma.log, ab_r02f_hybrid.log).  The traversal is bound by the
// latency of its scattered node fetches at 8 warps per scheduler, not by its instruction count.
#ifndef RRS_TRAV_FMA
#define RRS_TRAV_FMA 0
#endif
struct RayK {
    float3 o, d, idir;
#if RRS_TRAV_FMA
    float3 an, af;  // -(o/d) -/+ 2^-21 |o/d|: t_near = fma(plane, 1/d, an), t_far = fma(plane, 1/d, af)
#endif
    uint32_t selx, sely, selz;  // PRMT selectors: (near, far) = (lo, hi) or (hi, lo) by the sign of 1/d
    uint32_t origin_word;       // RRS_NO_PRIM, or primitive index | RRS_ORG64 (the ray carries an f64 origin)
};
struct Trav {
    uint32_t cur;   // node index, leaf run reference, or TRAV_DONE
    uint32_t sp;    // stack entries in use (>= 1: the sentinel)
    float tbest;
    uint32_t best;
};

// prmt.b32 without the selector mask __byte_perm adds (3 LOP3 per node step)
__device__ __forceinline__ uint32_t prmt(uint32_t a, uint32_t sel) {
    uint32_t r;
    asm("prmt.b32 %0, %1, 0, %2;" : "=r"(r) : "r"(a), "r"(sel));
    return r;
}

__device__ __forceinline__ void trav_begin(const DScene& sc, float3 o, float3 d, uint32_t origin_word, const SStack& stack,
                                           RayK& r, Trav& tv) {
    r.o = o;
    r.d = d;
    r.idir = f3(1.0f / d.x, 1.0f / d.y, 1.0f / d.z);
    r.origin_word = origin_word;
#if RRS_TRAV_FMA
    {
        const float3 op = f3(o.x * r.idir.x, o.y * r.idir.y, o.z * r.idir.z);
        const float k = 4.76837158e-7f;  // 2^-21
        r.an = f3(-op.x - fabsf(op.x) * k, -op.y - fabsf(op.y) * k, -op.z - fabsf(op.z) * k);
        r.af = f3(-op.x + fabsf(op.x) * k, -op.y + fabsf(op.y) * k, -op.z + fabsf(op.z) * k);
    }
#endif
    r.selx = r.idir.x < 0.f ? 0x1032u : 0x3210u;
    r.sely = r.idir.y < 0.f ? 0x1032u : 0x3210u;
    r.selz = r.idir.z < 0.f ? 0x1032u : 0x3210u;
    stack.set(0u, TRAV_DONE);
    tv.cur = sc.root;
    tv.sp = 1;
    tv.tbest = sc.tmax;
    tv.best = RRS_NO_PRIM;
}

__device__ __forceinline__ bool trav_on_inner(const Trav& tv) { return (int32_t)tv.cur >= 0; }
__device__ __forceinline__ __half2 u32_as_half2(uint32_t v) { return *reinterpret_cast<__half2*>(&v); }

// (p - o) * i for both planes p of one axis in paired FP32 (sub.rn.f32x2 / mul.rn.f32x2: IEEE round-to-nearest per
// half, denormals kept — no .ftz, as the scalar form).
__device__ __forceinline__ void slab2(float2 p, float o, float i, float& t0, float& t1) {
    unsigned long long v;
    asm("{\n\t.reg .b64 po, pi;\n\t"
        "mov.b64 po, {%3, %3};\n\t"
        "mov.b64 pi, {%4, %4};\n\t"
        "mov.b64 %0, {%1, %2};\n\t"
        "sub.rn.f32x2 %0, %0, po;\n\t"
        "mul.rn.f32x2 %0, %0, pi;\n\t}"
        : "=&l"(v) : "f"(p.x), "f"(p.y), "f"(o), "f"(i));
    asm("mov.b64 {%0, %1}, %2;" : "=f"(t0), "=f"(t1) : "l"(v));
}
// One inner node: both child boxes from one 2 x 256-bit fetch, near child first, far child pushed.
template <bool COUNT>
__device__ __forceinline__ void trav_node_step(const DScene& sc, const RayK& r, Trav& tv, const SStack& stack,
                                               TravCounters& cnt) {
    uint32_t w[8];
    RRS_CHECK(tv.cur < sc.n_nodes);
    ldg256(sc.nodes + tv.cur, w);
    if (COUNT) cnt.nodes++;
    const float3 idir = r.idir;
    const uint32_t ref0 = w[6], ref1 = w[7];
    // (Requesting BOTH children's records here — prefetch.global.L1 the moment their references arrive, so that the box
    // tests below cover the fetch the next step depends on — halves the speed: -45 % on configurations 4 and 5,
    // profiles/ab_logs/ab_r02p_prefetch.log.  The loop is bound by the rate at which L1 accepts scattered 32-byte
    // requests, one tag lookup per lane per node, not by the latency of any single one.)
    // Slab test as geometry.rs:458-513 writes it: the near/far plane is chosen by the sign of
    // 1/d (not by min/max of the two products), and max/min drop NaNs — so a ray lying in a
    // face plane of the box (0 * inf = NaN) is simply not constrained by that axis.
    // (selectors rebuilt here from the sign bits of 1/d — three registers fewer per ray — measured +-0:
    // profiles/ab_logs/ab_r02l_regs.log)
    const uint32_t selx = r.selx, sely = r.sely, selz = r.selz;
    const float2 ax = __half22float2(u32_as_half2(prmt(w[0], selx)));  // (near, far) planes
    const float2 ay = __half22float2(u32_as_half2(prmt(w[1], sely)));
    const float2 az = __half22float2(u32_as_half2(prmt(w[2], selz)));
    const float2 bx = __half22float2(u32_as_half2(prmt(w[3], selx)));
    const float2 by = __half22float2(u32_as_half2(prmt(w[4], sely)));
    const float2 bz = __half22float2(u32_as_half2(prmt(w[5], selz)));
#if RRS_TRAV_FMA
    const float3 an = r.an, af = r.af;
    float ax0 = fmaf(ax.x, idir.x, an.x), ax1 = fmaf(ax.y, idir.x, af.x);
    float ay0 = fmaf(ay.x, idir.y, an.y), ay1 = fmaf(ay.y, idir.y, af.y);
    float az0 = fmaf(az.x, idir.z, an.z), az1 = fmaf(az.y, idir.z, af.z);
    float bx0 = fmaf(bx.x, idir.x, an.x), bx1 = fmaf(bx.y, idir.x, af.x);
    float by0 = fmaf(by.x, idir.y, an.y), by1 = fmaf(by.y, idir.y, af.y);
    float bz0 = fmaf(bz.x, idir.z, an.z), bz1 = fmaf(bz.y, idir.z, af.z);
#else
    // (near, far) of one axis as one pair: (plane - o) * (1/d) in paired FP32 (FADD2 + FMUL2, o and 1/d broadcast),
    // each half rounded as the scalar FADD / FMUL it replaces (a product of a difference cannot contract into an FMA):
    // bitwise the same distances as the scalar form, 6 instructions per child instead of 12.  (The max / min chains
    // below compile to 3-input FMNMX as they are.)
    const float3 o = r.o;
    float ax0, ax1, ay0, ay1, az0, az1, bx0, bx1, by0, by1, bz0, bz1;
    slab2(ax, o.x, idir.x, ax0, ax1);
    slab2(ay, o.y, idir.y, ay0, ay1);
    slab2(az, o.z, idir.z, az0, az1);
    slab2(bx, o.x, idir.x, bx0, bx1);
    slab2(by, o.y, idir.y, by0, by1);
    slab2(bz, o.z, idir.z, bz0, bz1);
#endif
    float n0 = fmaxf(fmaxf(ax0, ay0), fmaxf(az0, sc.tmin));
    float f0 = fminf(fminf(ax1, ay1), fminf(az1, tv.tbest));
    float n1 = fmaxf(fmaxf(bx0, by0), fmaxf(bz0, sc.tmin));
    float f1 = fminf(fminf(bx1, by1), fminf(bz1, tv.tbest));
    // conservative acceptance: fp32 slab arithmetic is good to a few ulp, boxes are
    // rounded outward, so anything the f64 test accepts is accepted here.  An RRS_REF_EMPTY child carries
    // an inverted infinite box (enforced at scene creation) and fails the test by itself.
    const bool go0 = n0 <= f0 * 1.000001f;
    const bool go1 = n1 <= f1 * 1.000001f;
    if (go0 && go1) {
        const bool swap = n1 < n0;
        RRS_CHECK(tv.sp < sc.stack_entries);
        stack.set(tv.sp, swap ? ref0 : ref1);
        ++tv.sp;
        tv.cur = swap ? ref1 : ref0;
    } else if (go0 || go1) {
        tv.cur = go0 ? ref0 : ref1;
    } else {
        RRS_CHECK(tv.sp >= 1u);
        --tv.sp;
        tv.cur = stack.get(tv.sp);
    }
}

// One primitive against the ray; RayIntersection::update (bvh.rs:50-72) on a hit.
template <bool SPH64>
__device__ __forceinline__ void test_prim(const DScene& sc, uint32_t pi, float4 a, float4 b, float4 c, float3 o, float3 d,
                                          const RayProj& proj, uint32_t origin_prim, const double* org64, float& tbest,
                                          uint32_t& best) {
    const uint32_t type = prim_type(a);
    float t;
    bool hit;
    if (type == RRS_TRIANGLE) {
        if (pi == origin_prim) return;  // planar primitive cannot re-hit itself
        hit = hit_triangle(a, b, c, o, d, proj, t);
    } else if (type == RRS_SPHERE) {
        if (SPH64 && pi == origin_prim && org64 != nullptr) {
            // re-entry: the reference's f64 arithmetic on the f64 hit point, then the leaf filter of bvh.rs:404-413 in f64
            hit = sphere_reentry64(sc, __float_as_uint(b.y), org64, d, &t);
        } else {
            hit = hit_sphere(a, b, o, d, pi == origin_prim, t);
        }
    } else {
        if (pi == origin_prim) return;
        hit = hit_plane(a, b, o, d, t);
    }
    // leaf filter + RayIntersection::update: strictly smaller t wins; equal t keeps
    // the lower DFS index (ordered traversal may meet them in either order)
    if (hit && t > sc.tmin && (t < tbest || (t == tbest && best != RRS_NO_PRIM && pi < best))) {
        tbest = t;
        best = pi;
    }
}

// Software pipelining of the leaf loop (record k + 1 fetched while record k is tested) held 12 more registers across
// the primitive test; without it the kernel spills less and runs 4 % faster on configurations 4 and 5
// (profiles/ab_logs/ab_r02k_leafpf.log) — the opposite of round 1's measurement, taken before the kernel was this
// close to its register limit.
#ifndef RRS_LEAF_PREFETCH
#define RRS_LEAF_PREFETCH 0
#endif
// One leaf run (1..4 primitives, DFS order), then pop.  org64: the f64 origin slot of THIS ray in the queue (SPH64).
template <bool COUNT, bool SPH64>
__device__ __forceinline__ void trav_leaf_step(const DScene& sc, const RayK& r, Trav& tv, const SStack& stack,
                                               const double* org64, TravCounters& cnt) {
    const uint32_t first = tv.cur & 0x0FFFFFFFu;
    const uint32_t count = ((tv.cur >> 28) & 7u) + 1u;
    // software-pipelined: the record of primitive k + 1 is in flight while primitive k is tested (the loads of a
    // run are independent of the tests, but the loop-carried closest hit keeps the compiler from hoisting them)
    float4 a, b, c, pad;
    RRS_CHECK(first + count <= sc.n_prims && tv.sp >= 1u);
    ldg256(sc.prims + first, a, b);
    ldg256(reinterpret_cast<const char*>(sc.prims + first) + 32, c, pad);
    // the shear rows are rebuilt per leaf visit (~3.5 per ray) instead of living in 6 registers for the
    // whole traversal (~30 node steps per ray); they overlap the first fetch
    const float3 o = r.o, d = r.d;
    const uint32_t origin_word = r.origin_word;
    const uint32_t origin_prim = origin_word == RRS_NO_PRIM ? RRS_NO_PRIM : (origin_word & RRS_PRIM_MASK);
    const double* o64 = (SPH64 && origin_word != RRS_NO_PRIM && (origin_word & RRS_ORG64)) ? org64 : nullptr;
    RayProj proj;
    if (sc.has_triangles) proj = make_proj(d);
#if RRS_LEAF_PREFETCH
    for (uint32_t k = 0; k < count; ++k) {
        const uint32_t pi = first + k;
        float4 na = a, nb = b, nc = c;
        if (k + 1 < count) {
            ldg256(sc.prims + pi + 1, na, nb);
            ldg256(reinterpret_cast<const char*>(sc.prims + pi + 1) + 32, nc, pad);
        }
        if (COUNT) cnt.prims++;
        test_prim<SPH64>(sc, pi, a, b, c, o, d, proj, origin_prim, o64, tv.tbest, tv.best);
        a = na;
        b = nb;
        c = nc;
    }
#else
    for (uint32_t pi = first, end = first + count;;) {
        if (COUNT) cnt.prims++;
        test_prim<SPH64>(sc, pi, a, b, c, o, d, proj, origin_prim, o64, tv.tbest, tv.best);
        if (++pi == end) break;
        ldg256(sc.prims + pi, a, b);
        ldg256(reinterpret_cast<const char*>(sc.prims + pi) + 32, c, pad);
    }
#endif
    --tv.sp;
    tv.cur = stack.get(tv.sp);
}

// Small scenes (<= RRS_BRUTE_MAX reachable primitives, every sphere-series configuration): the BVH is
// pure overhead — its two or three node steps cost as much as the tests they save and de-synchronise
// the lanes.  All reachable primitives are tested instead, in DFS order, from a copy staged in shared
// memory (one broadcast LDS per record, no stack, no divergence: every lane runs the same loop).  Same
// result as the traversal: a box never rejects a ray that hits a primitive inside it, and primitives
// under a dead node (SURVEY.md F6) are not in the list.
// RayIntersection::update (bvh.rs:50-72) with the leaf filter of bvh.rs:404-413
__device__ __forceinline__ void update_hit(const DScene& sc, bool hit, float t, uint32_t pi, float& tbest, uint32_t& best) {
    if (hit && t > sc.tmin && (t < tbest || (t == tbest && best != RRS_NO_PRIM && pi < best))) {
        tbest = t;
        best = pi;
    }
}

// Conservative slab test of a ray against a box padded outward on the host (the sphere group of the brute-force list).
// min/max drop NaNs (a ray lying in a face plane of the padded box cannot reach what is strictly inside it); the
// reciprocal is the 1-ulp approximation and the products carry ~1e-7 relative error each, covered by the 1e-6 slack.
__device__ __forceinline__ float rcp_approx(float x) {
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
__device__ __forceinline__ bool ray_meets_box(const float* __restrict__ box, float3 o, float3 d) {
    const float ix = rcp_approx(d.x), iy = rcp_approx(d.y), iz = rcp_approx(d.z);
    const float x0 = (box[0] - o.x) * ix, x1 = (box[3] - o.x) * ix;
    const float y0 = (box[1] - o.y) * iy, y1 = (box[4] - o.y) * iy;
    const float z0 = (box[2] - o.z) * iz, z1 = (box[5] - o.z) * iz;
    const float tn = fmaxf(fmaxf(fminf(x0, x1), fminf(y0, y1)), fminf(z0, z1));
    const float tf = fminf(fminf(fmaxf(x0, x1), fmaxf(y0, y1)), fmaxf(z0, z1));
    return tf >= 0.f && tn <= tf * 1.000001f;
}

// The list is grouped by type on the host (spheres, planes, triangles; DFS order inside a group), so each group is a
// tight loop without a per-primitive type dispatch; the tie-break still goes by the DFS index each record carries.
template <bool COUNT, bool SPH64>
__device__ __forceinline__ void closest_hit_brute(const DScene& sc, const DPrim* __restrict__ s_prims, float3 o, float3 d,
                                                  uint32_t origin_word, const double* __restrict__ org64, float& tbest,
                                                  uint32_t& best, TravCounters& cnt) {
    const uint32_t origin_prim = origin_word == RRS_NO_PRIM ? RRS_NO_PRIM : (origin_word & RRS_PRIM_MASK);
    const double* o64 = (SPH64 && origin_word != RRS_NO_PRIM && (origin_word & RRS_ORG64)) ? org64 : nullptr;
    tbest = sc.tmax;
    best = RRS_NO_PRIM;
    if (COUNT) cnt.prims += sc.brute_count;
    if (SPH64) {
        // the f64 variants keep the generic loop: with the re-entry branch inside, the grouped form measured 9 % slower
        // on the frosted-glass series (gpurun_out/sweep_grouped.log)
        RayProj proj;
        if (sc.has_triangles) proj = make_proj(d);
        // the list starts with the sphere group: skip it when the ray misses the group's box
        const uint32_t j0 = (sc.brute_box_on && !ray_meets_box(sc.brute_box, o, d)) ? sc.brute_spheres : 0u;
        for (uint32_t j = j0; j < sc.brute_count; ++j) {
            const DPrim& p = s_prims[j];
            test_prim<SPH64>(sc, sc.brute_prim[j], p.a, p.b, p.c, o, d, proj, origin_prim, o64, tbest, best);
        }
        return;
    }
    uint32_t k = 0;
    if (sc.brute_box_on && !ray_meets_box(sc.brute_box, o, d)) k = sc.brute_spheres;  // no sphere can be hit
    for (; k < sc.brute_spheres; ++k) {
        const uint32_t pi = sc.brute_prim[k];
        const float4 a = s_prims[k].a, b = s_prims[k].b;
        float t;
        const bool hit = hit_sphere(a, b, o, d, pi == origin_prim, t);  // (the f64 re-entry variants took the loop above)
        update_hit(sc, hit, t, pi, tbest, best);
    }
    for (; k < sc.brute_spheres + sc.brute_planes; ++k) {
        const uint32_t pi = sc.brute_prim[k];
        float t = 0.f;
        const bool hit = pi != origin_prim && hit_plane(s_prims[k].a, s_prims[k].b, o, d, t);  // a planar primitive cannot re-hit itself
        update_hit(sc, hit, t, pi, tbest, best);
    }
    if (k < sc.brute_count) {
        const RayProj proj = make_proj(d);
        for (; k < sc.brute_count; ++k) {
            const uint32_t pi = sc.brute_prim[k];
            float t = 0.f;
            const bool hit = pi != origin_prim && hit_triangle(s_prims[k].a, s_prims[k].b, s_prims[k].c, o, d, proj, t);
            update_hit(sc, hit, t, pi, tbest, best);
        }
    }
}

// block-wide copy of the brute-force list into shared memory (call before the first __syncthreads)
__device__ __forceinline__ void stage_brute_prims(const DScene& sc, DPrim* s_prims) {
    const uint32_t n4 = sc.brute_count * 4u;
    for (uint32_t i = threadIdx.x; i < n4; i += blockDim.x) {
        const float4* src = reinterpret_cast<const float4*>(sc.prims + sc.brute_prim[i >> 2]) + (i & 3u);
        reinterpret_cast<float4*>(s_prims)[i] = __ldg(src);
    }
}

// Per-thread traversal to completion (parity probes; the render path batches the steps per warp).
template <bool COUNT, bool SPH64>
__device__ __forceinline__ void closest_hit(const DScene& sc, float3 o, float3 d, uint32_t origin_word,
                                            const double* __restrict__ org64, const SStack& stack, float& tbest,
                                            uint32_t& best, TravCounters& cnt) {
    RayK r;
    Trav tv;
    trav_begin(sc, o, d, origin_word, stack, r, tv);
    while (tv.cur != TRAV_DONE) {
        while (trav_on_inner(tv)) trav_node_step<COUNT>(sc, r, tv, stack, cnt);
        if (tv.cur != TRAV_DONE) trav_leaf_step<COUNT, SPH64>(sc, r, tv, stack, org64, cnt);
    }
    tbest = tv.tbest;
    best = tv.best;
}

// triangle_t64 for the closest hit `best` of a finished query (no-op for misses, spheres and planes)
__device__ __forceinline__ float refine_hit_t(const DScene& sc, uint32_t best, float3 o, float3 d, float t) {
    if (best == RRS_NO_PRIM || !sc.has_triangles) return t;
    const float4* pp = reinterpret_cast<const float4*>(sc.prims + best);
    const float4 a = __ldg(pp);
    if (prim_type(a) != RRS_TRIANGLE) return t;
    return triangle_t64(sc, best, a, __ldg(pp + 1), __ldg(pp + 2), o, d, t);
}

}  // namespace rrs
