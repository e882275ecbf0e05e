// C ABI of the backend (include/rayrs_b200.h): scene validation, fp32 conversion, upload,
// and the thin entry points over wavefront.cu / verify_f64.cu.
#include <algorithm>
#include <cstdlib>
#include <cmath>
#include <cstring>
#include <string>
#include <limits>
#include <mutex>
#include <thread>
#include <vector>

#include <cuda_fp16.h>

#include "wavefront.cuh"

using namespace rrs;


static thread_local std::string g_last_error;

static int fail(int code, const std::string& msg) {
    g_last_error = msg;
    return code;
}
namespace rrs {
int api_fail(int code, const std::string& msg) { return fail(code, msg); }  // multi.cu shares the error channel
}

static bool in01(const double* c) {
    for (int k = 0; k < 3; ++k)
        if (!(c[k] >= 0. && c[k] <= 1.)) return false;
    return true;
}

static int usable_devices() {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    int ok = 0;
    for (int d = 0; d < n; ++d) {
        cudaDeviceProp p;
        if (cudaGetDeviceProperties(&p, d) == cudaSuccess && p.major == 10 && p.minor == 0) ok++;
    }
    return ok;
}

// f(begin, end) over [0, n) on up to one thread per hardware thread: scene descriptions of millions of primitives are
// validated and converted on all host cores (the 4M-triangle scene: 0.5 s -> 0.1 s)
template <typename F>
static void parallel_chunks(size_t n, size_t min_chunk, F f) {
    size_t threads = std::max<size_t>(1, std::thread::hardware_concurrency());
    threads = std::min(threads, std::max<size_t>(1, n / std::max<size_t>(1, min_chunk)));
    if (threads <= 1) {
        f((size_t)0, n);
        return;
    }
    std::vector<std::thread> pool;
    for (size_t t = 0; t < threads; ++t) pool.emplace_back([=]() { f(n * t / threads, n * (t + 1) / threads); });
    for (auto& th : pool) th.join();
}

template <typename T>
static int upload(T** dst, const T* src, size_t n, std::string& err) {
    RRS_CUDA_CHECK(cudaMalloc(dst, sizeof(T) * std::max<size_t>(n, 1)), err);
    if (n) RRS_CUDA_CHECK(cudaMemcpy(*dst, src, sizeof(T) * n, cudaMemcpyHostToDevice), err);
    return RRS_OK;
}

extern "C" {

int rrs_abi_version(void) { return RRS_ABI_VERSION; }
const char* rrs_last_error(void) { return g_last_error.c_str(); }
int rrs_device_count(void) { return usable_devices(); }

// ---------------------------------------------------------------------------------------
// Scene::new, device half.  Three steps so that a scene replicated on n GPUs is validated and
// converted once: validate(desc) -> convert(desc) -> upload(device) x n.
// ---------------------------------------------------------------------------------------
namespace {

// Everything derived from the description on the host: the device records and the DScene fields that do not
// depend on device addresses.
struct HostScene {
    std::vector<DPrim> prims;
    std::vector<DNode16> nodes;
    std::vector<DMat> mats;
    std::vector<float4> emis;
    std::vector<float4> hdri;
    std::vector<double4> sphere64;  // exact sphere parameters (see "sphere re-entry" in intersect.cuh)
    bool transmissive_sphere = false;
    std::vector<double> tri64;  // 9 doubles per primitive index, only when a triangle vertex is not exact in fp32
    // environment sampling table (env.cuh): empty when the map is black; env_ok false when it cannot be tabulated
    std::vector<float> env_marg, env_cond;
    std::vector<float2> env_row;
    bool env_ok = true;
    DScene d{};  // pointer members are filled per device
};

// Steps of a CDF over n cells of weights w (sum > 0), in units of 2^-24, the resolution of the device's uniforms:
// proportional to w, at least one step for every positive cell, none for a zero cell, 2^24 in all.  Writes each
// cell's start (exact in fp32).  False if the positive cells are too many for 2^24 steps.
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
    k[big] += G - tot;  // rounding and the one-step minimum go to the largest cell
    if (k[big] < 1) return false;
    int64_t acc = 0;
    for (size_t j = 0; j < n; ++j) {
        start[j] = std::ldexp((float)acc, -24);
        acc += k[j];
    }
    return true;
}

// The sampling table of RRS_FLAG_ENV_SAMPLING (env.cuh): per cell between texel centres the largest max(|r|,|g|,|b|)
// of its 4 corners times its solid angle; the marginal CDF over rows and one conditional CDF per row.
// 4 bytes per cell + 8 per row on the device (a 2048 x 1024 map: 8.4 MB).
static void build_env_table(const std::vector<float4>& hdri, uint32_t w, uint32_t h, HostScene& out) {
    const uint32_t cw = w - 1, ch = h - 1;
    auto lum = [&](uint32_t i, uint32_t j) {
        const float4 t = hdri[(size_t)i * w + j];
        return std::max(std::fabs(t.x), std::max(std::fabs(t.y), std::fabs(t.z)));
    };
    std::vector<double> cell((size_t)cw * ch), rows(ch);
    out.env_row.resize(ch);
    const double dphi = 2. * M_PI / cw;
    double total = 0.;
    for (uint32_t i = 0; i < ch; ++i) {
        const double t0 = M_PI * i / ch, t1 = M_PI * (i + 1) / ch;
        const double dcos = 2. * std::sin(0.5 * (t0 + t1)) * std::sin(0.5 * (t1 - t0));  // cos t0 - cos t1
        out.env_row[i] = make_float2((float)std::cos(t0), (float)dcos);
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
    if (!std::isfinite(total)) {
        out.env_ok = false;
        return;
    }
    if (total == 0.) return;  // a black map: nothing to sample
    out.env_marg.resize(ch);
    out.env_cond.assign((size_t)cw * ch, 0.f);
    bool ok = quantize_cdf(rows.data(), ch, total, out.env_marg.data());
    for (uint32_t i = 0; i < ch && ok; ++i)
        if (rows[i] > 0.) ok = quantize_cdf(cell.data() + (size_t)i * cw, cw, rows[i], out.env_cond.data() + (size_t)i * cw);
    if (!ok) {
        out.env_ok = false;
        out.env_marg.clear();
        out.env_cond.clear();
    }
}

int validate_desc(const RrsSceneDesc* desc, std::string& err) {
    auto bad = [&](int code, const char* m) { err = m; return code; };
    if (desc->abi_version != RRS_ABI_VERSION) return bad(RRS_ERR_INVALID, "ABI version mismatch");
    // --- the reference's construction-time assert!s ----------------------------------------
    if (desc->n_prims == 0 || !desc->prims) return bad(RRS_ERR_INVALID, "a BVH for 0 objects does not make sense (bvh.rs:229)");
    if (desc->n_prims >= (1u << 28)) return bad(RRS_ERR_INVALID, "too many primitives (max 2^28-1)");
    if (desc->n_nodes == 0 || !desc->nodes) return bad(RRS_ERR_INVALID, "no BVH nodes");
    if (desc->n_nodes >= 0x80000000u) return bad(RRS_ERR_INVALID, "too many BVH nodes");
    if (!(desc->t_min >= 0.)) return bad(RRS_ERR_INVALID, "z_near must be >= 0 (lib.rs:234)");
    if (!(desc->t_max > desc->t_min)) return bad(RRS_ERR_INVALID, "z_far must be > z_near (lib.rs:235)");
    if (desc->n_materials == 0 || !desc->materials) return bad(RRS_ERR_INVALID, "no materials");
    if (desc->n_emissions > 0 && !desc->emissions) return bad(RRS_ERR_INVALID, "n_emissions > 0 but emissions is NULL");
    if (desc->hdri_width < 2 || desc->hdri_height < 2 || !desc->hdri_rgb) return bad(RRS_ERR_INVALID, "HDRI must be at least 2x2");
    if (desc->refill_lanes > 32) return bad(RRS_ERR_INVALID, "refill_lanes must be within 0..32");
    for (uint32_t i = 0; i < desc->n_materials; ++i) {
        const RrsMaterial& m = desc->materials[i];
        if (m.tag > RRS_MAT_NO_REFLECT) return bad(RRS_ERR_INVALID, "unknown material tag");
        if (m.tag == RRS_MAT_NO_REFLECT) continue;
        if (!in01(m.color)) return bad(RRS_ERR_INVALID, "material color must be within [0,1] (material.rs:597)");
        bool rough = m.tag == RRS_MAT_COOK_TORRANCE || m.tag == RRS_MAT_COOK_TORRANCE_REFRACT ||
                     m.tag == RRS_MAT_COOK_TORRANCE_GLASS || m.tag == RRS_MAT_PLASTIC;
        bool has_ior = m.tag == RRS_MAT_REFRACT || m.tag == RRS_MAT_GLASS || m.tag == RRS_MAT_COOK_TORRANCE_REFRACT ||
                       m.tag == RRS_MAT_COOK_TORRANCE_GLASS || m.tag == RRS_MAT_PLASTIC ||
                       (m.tag == RRS_MAT_COOK_TORRANCE && m.fresnel_kind == RRS_FRESNEL_DIELECTRIC);
        if (rough && !(m.alpha > 0. && std::isfinite(m.alpha))) return bad(RRS_ERR_INVALID, "alpha must be positive and finite (material.rs:706-707)");
        if (has_ior && !(m.ior > 0. && std::isfinite(m.ior))) return bad(RRS_ERR_INVALID, "ior must be positive and finite (material.rs:629-630)");
        if (m.tag == RRS_MAT_PLASTIC && !in01(m.spec_color)) return bad(RRS_ERR_INVALID, "spec_color must be within [0,1] (material.rs:882)");
        if (m.fresnel_kind > RRS_FRESNEL_METALLIC) return bad(RRS_ERR_INVALID, "unknown Fresnel kind");
    }
    for (uint32_t i = 0; i < desc->n_emissions; ++i) {
        if (!(desc->emissions[i].strength >= 0.)) return bad(RRS_ERR_INVALID, "emission strength must be >= 0 (material.rs:1064)");
        if (!in01(desc->emissions[i].color)) return bad(RRS_ERR_INVALID, "RGB values need to be between 0 and 1 (material.rs:1065-1068)");
    }
    {
        std::mutex mu;
        const char* first_error = nullptr;
        parallel_chunks(desc->n_prims, 1 << 16, [&](size_t lo, size_t hi) {
            const char* e = nullptr;
            for (size_t i = lo; i < hi && !e; ++i) {
                const RrsPrim& p = desc->prims[i];
                if (p.type > RRS_TRIANGLE) e = "unknown primitive type";
                else if (p.material >= desc->n_materials) e = "primitive material index out of range";
                else if (p.emission >= (int32_t)desc->n_emissions) e = "primitive emission index out of range";
                else if (p.type == RRS_SPHERE && !(p.v[0] > 0.)) e = "Radius has to be positive (geometry.rs:97)";
                else if (p.type == RRS_PLANE && !(p.v[0] >= 0. && p.v[0] <= 5.)) e = "unknown plane axis";
                else if (p.type == RRS_PLANE && !(p.v[1] < p.v[2] && p.v[3] < p.v[4]))
                    e = "Plane cannot be constructed with umin >= umax or vmin >= vmax (geometry.rs:205-212)";
                for (int k = 0; k < 9 && !e; ++k)
                    if (std::isnan(p.v[k])) e = "NaN in primitive (bvh.rs:104 partial_cmp().unwrap() panics)";
            }
            if (e) {
                std::lock_guard<std::mutex> g(mu);
                if (!first_error) first_error = e;
            }
        });
        if (first_error) return bad(RRS_ERR_INVALID, first_error);
    }
    for (uint32_t i = 0; i < desc->n_nodes; ++i) {
        const RrsNode& nd = desc->nodes[i];
        const uint32_t refs[2] = {nd.ref0, nd.ref1};
        for (uint32_t r : refs) {
            if (r == RRS_REF_EMPTY) continue;
            if (r & RRS_REF_LEAF) {
                uint32_t first = r & 0x0FFFFFFFu, count = ((r >> 28) & 7u) + 1u;
                if (count > 4 || first + count > desc->n_prims) return bad(RRS_ERR_INVALID, "leaf run out of range");
            } else if (r >= desc->n_nodes || r == 0) {
                return bad(RRS_ERR_INVALID, "node reference out of range");
            }
        }
    }
    // The traversal stack in shared memory is sized from max_depth and the release kernels do not bounds-check it,
    // so the value is not taken on trust: walk the node graph from node 0, reject a node reached twice (a cycle or
    // a DAG — neither is a tree, and a cycle would spin the persistent kernel forever) and a chain longer than stated.
    if (desc->max_depth > 117u) return bad(RRS_ERR_TOO_DEEP, "BVH deeper than the 117-entry shared-memory traversal stack");
    {
        std::vector<uint8_t> seen(desc->n_nodes, 0);
        std::vector<std::pair<uint32_t, uint32_t>> todo;  // (node, depth)
        todo.emplace_back(0u, 1u);
        seen[0] = 1;
        while (!todo.empty()) {
            const auto [f, depth] = todo.back();
            todo.pop_back();
            if (depth > desc->max_depth) return bad(RRS_ERR_INVALID, "BVH is deeper than RrsSceneDesc.max_depth states");
            for (uint32_t r : {desc->nodes[f].ref0, desc->nodes[f].ref1}) {
                if (r == RRS_REF_EMPTY || (r & RRS_REF_LEAF)) continue;
                if (seen[r]) return bad(RRS_ERR_INVALID, "BVH node reached twice: the node graph must be a tree (no cycles, no shared subtrees)");
                seen[r] = 1;
                todo.emplace_back(r, depth + 1u);
            }
        }
    }
    return RRS_OK;
}

void convert_desc(const RrsSceneDesc* desc, HostScene& h) {
    h.prims.resize(desc->n_prims);
    bool has_triangles = false, inexact_vertex = false;
    auto meta_of = [&](const RrsPrim& p, float& fmeta, float& fobj, float& femi) {
        const uint32_t meta = p.type | (p.material << 2);
        const int32_t emi = p.emission;
        std::memcpy(&fmeta, &meta, 4);
        std::memcpy(&fobj, &p.obj_id, 4);
        std::memcpy(&femi, &emi, 4);
    };
    {
        // triangles (the millions) on all host threads ...
        std::mutex mu;
        parallel_chunks(desc->n_prims, 1 << 16, [&](size_t lo, size_t hi) {
            bool tri = false, inexact = false;
            for (size_t i = lo; i < hi; ++i) {
                const RrsPrim& p = desc->prims[i];
                if (p.type != RRS_TRIANGLE) continue;
                tri = true;
                float fmeta, fobj, femi;
                meta_of(p, fmeta, fobj, femi);
                for (int k = 0; k < 9; ++k) inexact = inexact || (double)(float)p.v[k] != p.v[k];
                // the three vertices (shared vertices of a mesh must stay bit-identical across triangles
                // for the watertight test, so no per-triangle edge vectors are stored)
                DPrim q;
                q.a = make_float4((float)p.v[0], (float)p.v[1], (float)p.v[2], fmeta);
                q.b = make_float4((float)p.v[3], (float)p.v[4], (float)p.v[5], fobj);
                q.c = make_float4((float)p.v[6], (float)p.v[7], (float)p.v[8], femi);
                q.pad = make_float4(0.f, 0.f, 0.f, 0.f);
                h.prims[i] = q;
            }
            std::lock_guard<std::mutex> g(mu);
            has_triangles = has_triangles || tri;
            inexact_vertex = inexact_vertex || inexact;
        });
    }
    // ... spheres and planes in order: a sphere's slot in sphere64 is its rank among the spheres
    for (uint32_t i = 0; i < desc->n_prims; ++i) {
        const RrsPrim& p = desc->prims[i];
        if (p.type == RRS_TRIANGLE) continue;
        DPrim q;
        float fmeta, fobj, femi;
        meta_of(p, fmeta, fobj, femi);
        if (p.type == RRS_SPHERE) {
            uint32_t sidx = (uint32_t)h.sphere64.size();
            float fsidx;
            std::memcpy(&fsidx, &sidx, 4);
            h.sphere64.push_back(make_double4(p.v[1], p.v[2], p.v[3], p.v[0]));
            uint32_t tag = desc->materials[p.material].tag;
            if (tag == RRS_MAT_REFRACT || tag == RRS_MAT_GLASS || tag == RRS_MAT_COOK_TORRANCE_REFRACT ||
                tag == RRS_MAT_COOK_TORRANCE_GLASS)
                h.transmissive_sphere = true;
            q.a = make_float4((float)p.v[1], (float)p.v[2], (float)p.v[3], fmeta);
            q.b = make_float4((float)p.v[0], fsidx, 0.f, fobj);
            q.c = make_float4(0.f, 0.f, 0.f, femi);
        } else {
            uint32_t axis = (uint32_t)p.v[0];
            float faxis;
            std::memcpy(&faxis, &axis, 4);
            q.a = make_float4((float)p.v[5], (float)p.v[1], (float)p.v[2], fmeta);
            q.b = make_float4((float)p.v[3], (float)p.v[4], faxis, fobj);
            q.c = make_float4(0.f, 0.f, 0.f, femi);
        }
        q.pad = make_float4(0.f, 0.f, 0.f, 0.f);
        h.prims[i] = q;
    }
    if (inexact_vertex) {
        // the f64 vertices travel too: triangle_t64 (intersect.cuh) re-evaluates the accepted hit's distance from them
        h.tri64.assign((size_t)desc->n_prims * 9, 0.);
        for (uint32_t i = 0; i < desc->n_prims; ++i)
            if (desc->prims[i].type == RRS_TRIANGLE) std::memcpy(&h.tri64[(size_t)i * 9], desc->prims[i].v, 9 * sizeof(double));
    }
    h.mats.resize(desc->n_materials);
    for (uint32_t i = 0; i < desc->n_materials; ++i) {
        const RrsMaterial& m = desc->materials[i];
        float ftag, fkind;
        uint32_t kind = m.fresnel_kind;
        if (m.tag != RRS_MAT_COOK_TORRANCE) kind = RRS_FRESNEL_DIELECTRIC;
        std::memcpy(&ftag, &m.tag, 4);
        std::memcpy(&fkind, &kind, 4);
        double r0 = (1. - m.ior) / (1. + m.ior);  // schlick_scalar r0, material.rs:1476-1477 (symmetric in the two iors)
        r0 = r0 * r0;
        DMat d;
        d.m0 = make_float4((float)m.color[0], (float)m.color[1], (float)m.color[2], ftag);
        d.m1 = make_float4((float)m.spec_color[0], (float)m.spec_color[1], (float)m.spec_color[2], (float)(m.alpha * m.alpha));
        d.m2 = make_float4((float)m.ior, fkind, (float)r0, 0.f);
        h.mats[i] = d;
    }
    h.emis.resize(std::max<uint32_t>(desc->n_emissions, 1));
    for (uint32_t i = 0; i < desc->n_emissions; ++i) {
        const RrsEmission& e = desc->emissions[i];
        h.emis[i] = make_float4((float)(e.strength * e.color[0]), (float)(e.strength * e.color[1]), (float)(e.strength * e.color[2]), 0.f);
    }
    size_t ntex = (size_t)desc->hdri_width * desc->hdri_height;
    h.hdri.resize(ntex);
    for (size_t i = 0; i < ntex; ++i)
        h.hdri[i] = make_float4(desc->hdri_rgb[3 * i], desc->hdri_rgb[3 * i + 1], desc->hdri_rgb[3 * i + 2], 0.f);
    build_env_table(h.hdri, desc->hdri_width, desc->hdri_height, h);
    static_assert(sizeof(RrsNode) == 64, "RrsNode must be 64 bytes");
    static_assert(sizeof(RrsNodeF64) == 128, "RrsNodeF64 must be 128 bytes");
    {
        // device nodes: fp16 boxes rounded outward, one half2 (lo, hi) word per axis (device_types.cuh).
        // An RRS_REF_EMPTY child must fail the slab test by itself (the traversal does not look at the
        // reference before testing the box): it gets the inverted infinite box whatever the caller stored.
        auto pack = [](float lo, float hi) -> uint32_t {
            __half hl = __float2half_rd(lo), hh = __float2half_ru(hi);  // overflow -> +-inf: still conservative
            uint16_t bl, bh;
            std::memcpy(&bl, &hl, 2);
            std::memcpy(&bh, &hh, 2);
            return (uint32_t)bl | ((uint32_t)bh << 16);
        };
        h.nodes.resize(desc->n_nodes);
        parallel_chunks(desc->n_nodes, 1 << 16, [&](size_t lo, size_t hi) {
            for (size_t i = lo; i < hi; ++i) {
                const RrsNode& nd = desc->nodes[i];
                DNode16& q = h.nodes[i];
                for (int k = 0; k < 3; ++k) {
                    q.w[k] = nd.ref0 == RRS_REF_EMPTY ? pack(INFINITY, -INFINITY) : pack(nd.lo0[k], nd.hi0[k]);
                    q.w[3 + k] = nd.ref1 == RRS_REF_EMPTY ? pack(INFINITY, -INFINITY) : pack(nd.lo1[k], nd.hi1[k]);
                }
                q.w[6] = nd.ref0;
                q.w[7] = nd.ref1;
            }
        });
    }
    DScene& d = h.d;
    d.n_prims = desc->n_prims;
    d.n_nodes = desc->n_nodes;
    d.n_mats = desc->n_materials;
    d.hdri_w = desc->hdri_width;
    d.hdri_h = desc->hdri_height;
    d.tmin = (float)desc->t_min;
    d.tmax = (float)desc->t_max;
    d.tmin64 = desc->t_min;
    d.tmax64 = desc->t_max;
    d.stack_entries = std::max<uint32_t>(desc->max_depth + 3, 4);  // + the TRAV_DONE sentinel
    d.has_triangles = has_triangles ? 1u : 0u;
    {
        // primitives the traversal can reach (leaf runs below live nodes), for the small-scene path
        std::vector<uint32_t> reach;
        std::vector<uint32_t> todo{0u};
        bool small = true;
        while (!todo.empty() && small) {
            const RrsNode& nd = desc->nodes[todo.back()];
            todo.pop_back();
            for (uint32_t r : {nd.ref0, nd.ref1}) {
                if (r == RRS_REF_EMPTY) continue;
                if (r & RRS_REF_LEAF) {
                    for (uint32_t k = 0; k <= ((r >> 28) & 7u); ++k) reach.push_back((r & 0x0FFFFFFFu) + k);
                } else {
                    todo.push_back(r);
                }
            }
            small = reach.size() <= RRS_BRUTE_MAX && todo.size() <= 64;
        }
        std::sort(reach.begin(), reach.end());
        reach.erase(std::unique(reach.begin(), reach.end()), reach.end());
        d.brute_count = 0;
        if (small && !reach.empty() && !(desc->flags & RRS_SCENE_NO_BRUTE)) {
            d.brute_count = (uint32_t)reach.size();
            // grouped by type (spheres, planes, triangles), DFS order inside a group
            std::stable_sort(reach.begin(), reach.end(), [&](uint32_t x, uint32_t y) {
                auto rank = [&](uint32_t i) { return desc->prims[i].type == RRS_SPHERE ? 0 : (desc->prims[i].type == RRS_PLANE ? 1 : 2); };
                return rank(x) < rank(y);
            });
            d.brute_spheres = d.brute_planes = 0;
            for (size_t k = 0; k < reach.size(); ++k) {
                d.brute_prim[k] = reach[k];
                if (desc->prims[reach[k]].type == RRS_SPHERE) d.brute_spheres++;
                else if (desc->prims[reach[k]].type == RRS_PLANE) d.brute_planes++;
            }
            // one box around the sphere group: a ray that misses it skips every sphere test (a one-level hierarchy;
            // most camera rays of the sphere-row scenes go to the floor or the sky).  Padded outward, so the fp32
            // slab test in closest_hit_brute stays conservative.
            d.brute_box_on = 0;
            if (d.brute_spheres >= 3) {
                double lo[3] = {1e300, 1e300, 1e300}, hi[3] = {-1e300, -1e300, -1e300};
                for (uint32_t k = 0; k < d.brute_spheres; ++k) {
                    const RrsPrim& p = desc->prims[reach[k]];
                    const double r = std::sqrt(p.v[0]);
                    for (int a = 0; a < 3; ++a) {
                        lo[a] = std::min(lo[a], p.v[1 + a] - r);
                        hi[a] = std::max(hi[a], p.v[1 + a] + r);
                    }
                }
                bool finite = true;
                for (int a = 0; a < 3; ++a) {
                    const double pad = 1e-5 * (hi[a] - lo[a]) + 1e-6 * std::max(std::fabs(lo[a]), std::fabs(hi[a])) + 1e-30;
                    d.brute_box[a] = std::nextafter((float)(lo[a] - pad), -std::numeric_limits<float>::infinity());
                    d.brute_box[3 + a] = std::nextafter((float)(hi[a] + pad), std::numeric_limits<float>::infinity());
                    finite = finite && std::isfinite(d.brute_box[a]) && std::isfinite(d.brute_box[3 + a]);
                }
                d.brute_box_on = (finite && !(desc->flags & RRS_SCENE_NO_BRUTE_BOX)) ? 1u : 0u;
            }
        }
    }
    {
        // children of the reference root lie inside its box, so its own slab test (the virtual root's
        // only job) can be skipped whenever the root is an inner node
        const RrsNode& vr = desc->nodes[0];
        d.root = (vr.ref1 == RRS_REF_EMPTY && vr.ref0 != RRS_REF_EMPTY && !(vr.ref0 & RRS_REF_LEAF)) ? vr.ref0 : 0u;
    }
    // rays of a deep tree differ widely in length: refill early; a tiny scene amortises the fetch over more lanes
    // (deep trees: 2 / 4 / 6 / 8 / 12 / 16 idle lanes measured, 8 is +1 % over round 1's 4: profiles/ab_logs/ab_r02u_refill.log)
    d.refill_lanes = desc->refill_lanes ? desc->refill_lanes : (desc->max_depth > 6 ? 8u : 12u);
}

int upload_scene(const RrsSceneDesc* desc, const HostScene& h, int device, RrsScene** out, std::string& err) {
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        err = "no CUDA device: rayrs_b200 has no CPU fallback";
        return RRS_ERR_NO_DEVICE;
    }
    if (device < 0 || device >= ndev) { err = "device index out of range"; return RRS_ERR_INVALID; }
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) { err = "cudaGetDeviceProperties failed"; return RRS_ERR_CUDA; }
    if (!(prop.major == 10 && prop.minor == 0)) {
        // the library holds sm_100a code only: an architecture-specific cubin has no PTX fallback and loads on 10.0 parts alone
        err = std::string("device is not sm_100 (") + prop.name + "): kernels are built for sm_100a only";
        return RRS_ERR_NO_DEVICE;
    }
    if (cudaSetDevice(device) != cudaSuccess) { err = "cudaSetDevice failed"; return RRS_ERR_CUDA; }

    auto* sc = new RrsScene();
    SceneImpl& s = sc->impl;
    s.device = device;
    s.num_sms = prop.multiProcessorCount;
    s.n_prims = desc->n_prims;
    s.n_nodes = desc->n_nodes;
    s.max_depth = desc->max_depth;
    s.tmin = desc->t_min;
    s.tmax = desc->t_max;
    int rc = RRS_OK;
    {
        // nodes and primitives share ONE allocation (nodes first) so that a single L2 access-policy window can
        // cover what the traversal fetches (wavefront.cu, "L2 residency")
        const size_t node_bytes = (sizeof(DNode16) * h.nodes.size() + 255) & ~(size_t)255;
        const size_t prim_bytes = sizeof(DPrim) * h.prims.size();
        auto up = [&]() -> int {
            RRS_CUDA_CHECK(cudaMalloc(&s.geom_blob, node_bytes + prim_bytes), err);
            RRS_CUDA_CHECK(cudaMemcpy(s.geom_blob, h.nodes.data(), sizeof(DNode16) * h.nodes.size(), cudaMemcpyHostToDevice), err);
            RRS_CUDA_CHECK(cudaMemcpy(s.geom_blob + node_bytes, h.prims.data(), prim_bytes, cudaMemcpyHostToDevice), err);
            return RRS_OK;
        };
        rc = up();
        s.nodes = reinterpret_cast<DNode16*>(s.geom_blob);
        s.prims = reinterpret_cast<DPrim*>(s.geom_blob + node_bytes);
        s.node_bytes = node_bytes;
        s.geom_bytes = node_bytes + prim_bytes;
    }
    if (rc == RRS_OK) rc = upload(&s.mats, h.mats.data(), h.mats.size(), err);
    if (rc == RRS_OK) rc = upload(&s.emis, h.emis.data(), h.emis.size(), err);
    if (rc == RRS_OK) rc = upload(&s.hdri, h.hdri.data(), h.hdri.size(), err);
    if (rc == RRS_OK && !h.env_marg.empty()) {
        float* marg = nullptr;
        float* cond = nullptr;
        float2* row = nullptr;
        rc = upload(&marg, h.env_marg.data(), h.env_marg.size(), err);
        s.env.marg = marg;
        if (rc == RRS_OK) rc = upload(&cond, h.env_cond.data(), h.env_cond.size(), err);
        s.env.cond = cond;
        if (rc == RRS_OK) rc = upload(&row, h.env_row.data(), h.env_row.size(), err);
        s.env.row = row;
    }
    s.env.cw = desc->hdri_width - 1;
    s.env.ch = desc->hdri_height - 1;
    s.env.inv_dphi = (float)(s.env.cw / (2. * M_PI));
    s.env_ok = h.env_ok;
    if (rc == RRS_OK && h.transmissive_sphere) rc = upload(&s.sphere64, h.sphere64.data(), h.sphere64.size(), err);
    if (rc == RRS_OK && !h.tri64.empty()) rc = upload(&s.tri64, h.tri64.data(), h.tri64.size(), err);
    if (rc == RRS_OK && desc->nodes_f64) {
        rc = upload(&s.nodes_f64, desc->nodes_f64, desc->n_nodes, err);
        if (rc == RRS_OK) rc = upload(&s.prims_f64, desc->prims, desc->n_prims, err);
    }
    if (rc == RRS_OK && !(desc->flags & RRS_SCENE_NO_L2_PERSIST)) {
        // L2 residency: how much of L2 the device lets a process set aside for persisting lines, and the largest
        // access-policy window.  The set-aside itself follows the RENDER (wf_render_accumulate): a render of the BVH
        // form claims it and pins the node (+ primitive) array through a window on its stream; a render of the
        // small-scene form hands it back — the carve-out is device-wide, and left in place it took 60 % of L2 away from
        // the queues of scenes that have no tree to pin (glass series -12 … -26 %, profiles/ab_logs/l2limit_r02v_c3.log).
        int max_persist = 0, max_window = 0;
        cudaDeviceGetAttribute(&max_persist, cudaDevAttrMaxPersistingL2CacheSize, device);
        cudaDeviceGetAttribute(&max_window, cudaDevAttrMaxAccessPolicyWindowSize, device);
        if (max_persist > 0 && max_window > 0) {
            s.l2_persist_bytes = (size_t)max_persist;
            s.l2_window_max = (size_t)max_window;
        }
        cudaGetLastError();
    }
    if (rc != RRS_OK) {
        rrs_scene_destroy(sc);
        return rc;
    }
    s.d = h.d;
    s.d.prims = s.prims;
    s.d.nodes = s.nodes;
    s.d.mats = s.mats;
    s.d.emis = s.emis;
    s.d.hdri = s.hdri;
    s.d.sphere64 = s.sphere64;
    s.d.tri64 = s.tri64;
    *out = sc;
    return RRS_OK;
}

}  // namespace

int rrs_scene_create(const RrsSceneDesc* desc, int device, RrsScene** out) {
    return rrs_scene_create_multi(desc, &device, 1, out);
}

int rrs_scene_create_multi(const RrsSceneDesc* desc, const int* devices, int n, RrsScene** out) {
    if (!desc || !out || !devices || n < 1) return fail(RRS_ERR_INVALID, "null argument");
    for (int i = 0; i < n; ++i) out[i] = nullptr;
    std::string err;
    int rc = validate_desc(desc, err);
    if (rc != RRS_OK) return fail(rc, err);
    // a host without any CUDA device fails before the conversion work
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return fail(RRS_ERR_NO_DEVICE, "no CUDA device: rayrs_b200 has no CPU fallback");
    }
    HostScene h;
    convert_desc(desc, h);
    for (int i = 0; i < n; ++i) {
        rc = upload_scene(desc, h, devices[i], &out[i], err);
        if (rc != RRS_OK) {
            for (int k = 0; k < i; ++k) {
                rrs_scene_destroy(out[k]);
                out[k] = nullptr;
            }
            return fail(rc, err);
        }
    }
    return RRS_OK;
}

void rrs_scene_destroy(RrsScene* scene) {
    if (!scene) return;
    SceneImpl& s = scene->impl;
    cudaSetDevice(s.device);
    wf_free(&s);
    cudaFree(s.geom_blob); cudaFree(s.mats); cudaFree(s.emis); cudaFree(s.hdri);
    cudaFree(const_cast<float*>(s.env.marg)); cudaFree(const_cast<float*>(s.env.cond)); cudaFree(const_cast<float2*>(s.env.row));
    cudaFree(s.prims_f64); cudaFree(s.nodes_f64); cudaFree(s.sphere64); cudaFree(s.tri64); cudaFree(s.accum); cudaFree(s.census); cudaFree(s.resolve_dev);
    if (s.resolve_pinned) cudaFreeHost(s.resolve_pinned);
    if (s.h_census) cudaFreeHost(s.h_census);
    if (s.own_stream) cudaStreamDestroy(s.own_stream);
    delete scene;
}

int rrs_render_accumulate(RrsScene* scene, const RrsCamera* camera, const RrsRenderParams* params, void* d_sum_rgba,
                          void* cuda_stream) {
    if (!scene) return fail(RRS_ERR_INVALID, "null scene");
    std::string err;
    int rc = wf_render_accumulate(&scene->impl, camera, params, static_cast<float4*>(d_sum_rgba),
                                  static_cast<cudaStream_t>(cuda_stream), err);
    return rc == RRS_OK ? rc : fail(rc, err);
}

int rrs_resolve(RrsScene* scene, const void* d_sum_rgba, uint32_t width, uint32_t height, uint32_t spp_total, float* out_rgb,
                int out_is_device, void* cuda_stream) {
    if (!scene) return fail(RRS_ERR_INVALID, "null scene");
    std::string err;
    int rc = wf_resolve(&scene->impl, static_cast<const float4*>(d_sum_rgba), width, height, spp_total, out_rgb,
                        out_is_device != 0, static_cast<cudaStream_t>(cuda_stream), err);
    return rc == RRS_OK ? rc : fail(rc, err);
}

int rrs_to_raw_bytes(RrsScene* scene, const void* d_sum_rgba, uint32_t width, uint32_t height, uint32_t spp_total,
                     double gamma, uint8_t* out_rgb8, int out_is_device, void* cuda_stream, uint64_t* census3) {
    if (!scene) return fail(RRS_ERR_INVALID, "null scene");
    std::string err;
    int rc = wf_to_raw_bytes(&scene->impl, static_cast<const float4*>(d_sum_rgba), width, height, spp_total, gamma, out_rgb8,
                             out_is_device != 0, static_cast<cudaStream_t>(cuda_stream), census3, err);
    return rc == RRS_OK ? rc : fail(rc, err);
}

int rrs_render(RrsScene* scene, const RrsCamera* camera, const RrsRenderParams* params, float* out_rgb) {
    if (!scene || !camera || !params || !out_rgb) return fail(RRS_ERR_INVALID, "null argument");
    SceneImpl& s = scene->impl;
    std::string err;
    if (cudaSetDevice(s.device) != cudaSuccess) return fail(RRS_ERR_CUDA, "cudaSetDevice failed");
    size_t npix = (size_t)params->width * params->height;
    if (npix == 0) return fail(RRS_ERR_INVALID, "empty image");
    if (s.accum_pixels != npix) {
        cudaFree(s.accum);
        s.accum = nullptr;
        if (cudaMalloc(&s.accum, sizeof(float4) * npix) != cudaSuccess) return fail(RRS_ERR_NOMEM, "cudaMalloc(accumulator) failed");
        s.accum_pixels = npix;
    }
    if (cudaMemsetAsync(s.accum, 0, sizeof(float4) * npix, nullptr) != cudaSuccess) return fail(RRS_ERR_CUDA, "cudaMemsetAsync failed");
    int rc = wf_render_accumulate(&s, camera, params, s.accum, nullptr, err);
    if (rc != RRS_OK) return fail(rc, err);
    uint64_t launches = s.stats.kernel_launches;
    uint32_t div = params->spp_total ? params->spp_total : params->spp;
    if (div == 0) div = 1;
    rc = wf_resolve(&s, s.accum, params->width, params->height, div, out_rgb, false, nullptr, err);
    if (rc != RRS_OK) return fail(rc, err);
    s.stats.kernel_launches = launches + 1;
    return RRS_OK;
}

int rrs_intersect(RrsScene* scene, const RrsRay* rays, size_t n, int32_t* obj_id, double* t, int precision) {
    if (!scene || (n && (!rays || !obj_id || !t))) return fail(RRS_ERR_INVALID, "null argument");
    std::string err;
    int rc;
    if (precision == 32) rc = wf_intersect32(&scene->impl, rays, n, obj_id, t, err);
    else if (precision == 64) rc = vf_intersect64(&scene->impl, rays, n, obj_id, t, err);
    else return fail(RRS_ERR_INVALID, "precision must be 32 or 64");
    return rc == RRS_OK ? rc : fail(rc, err);
}

int rrs_material_evaluate(RrsScene* scene, uint32_t material, const double* normal_view, const double* u, size_t n,
                          float* out) {
    if (!scene || (n && (!normal_view || !u || !out))) return fail(RRS_ERR_INVALID, "null argument");
    std::string err;
    int rc = wf_material_evaluate(&scene->impl, material, normal_view, u, n, out, err);
    return rc == RRS_OK ? rc : fail(rc, err);
}

int rrs_material_evaluate_pdf(RrsScene* scene, uint32_t material, const RrsPrim* light, const double* pos_normal_view,
                              const double* u, size_t n, double* out) {
    if (!scene || !light || (n && (!pos_normal_view || !u || !out))) return fail(RRS_ERR_INVALID, "null argument");
    std::string err;
    int rc = nee_material_evaluate_pdf(&scene->impl, material, light, pos_normal_view, u, n, out, err);
    return rc == RRS_OK ? rc : fail(rc, err);
}

int rrs_background(RrsScene* scene, const double* dirs, size_t n, float* out) {
    if (!scene || (n && (!dirs || !out))) return fail(RRS_ERR_INVALID, "null argument");
    std::string err;
    int rc = wf_background(&scene->impl, dirs, n, out, err);
    return rc == RRS_OK ? rc : fail(rc, err);
}

int rrs_env_sample(RrsScene* scene, const double* u, size_t n, double* dir_pdf) {
    if (!scene || (n && (!u || !dir_pdf))) return fail(RRS_ERR_INVALID, "null argument");
    std::string err;
    int rc = wf_env_sample(&scene->impl, u, n, dir_pdf, err);
    return rc == RRS_OK ? rc : fail(rc, err);
}

int rrs_env_pdf(RrsScene* scene, const double* dirs, size_t n, double* pdf) {
    if (!scene || (n && (!dirs || !pdf))) return fail(RRS_ERR_INVALID, "null argument");
    std::string err;
    int rc = wf_env_pdf(&scene->impl, dirs, n, pdf, err);
    return rc == RRS_OK ? rc : fail(rc, err);
}

int rrs_rng_uniforms(RrsScene* scene, uint64_t seed, uint32_t pixel, uint32_t sample, uint32_t slot, float* out4) {
    if (!scene || !out4) return fail(RRS_ERR_INVALID, "null argument");
    std::string err;
    int rc = wf_rng_uniforms(&scene->impl, seed, pixel, sample, slot, out4, err);
    return rc == RRS_OK ? rc : fail(rc, err);
}

int rrs_stats(RrsScene* scene, RrsStats* out) {
    if (!scene || !out) return fail(RRS_ERR_INVALID, "null argument");
    wf_finish_stats(&scene->impl);  // waits for an asynchronous rrs_render_accumulate
    *out = scene->impl.stats;
    return RRS_OK;
}

}  // extern "C"
