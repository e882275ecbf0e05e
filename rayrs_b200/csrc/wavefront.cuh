// Wavefront path-tracing state shared between wavefront.cu (kernels + render loop) and
// api.cu (scene handle).
#pragma once
#include <cuda_runtime.h>

#include <string>
#include <vector>

#include "device_types.cuh"
#include "env.cuh"

namespace rrs {

// Device-resident loop state.  Everything the persistent kernels need to size their work is
// read from here, so an iteration needs no host round trip.
struct DCounters {
    uint32_t n_cur;       // rays in the current queue (extend + shade work size)
    uint32_t n_next;      // survivors appended to the other queue by shade
    uint32_t gen_count;   // padded path indices to generate this iteration
    uint32_t done;        // 1 when no live ray and no path left
    unsigned long long gen_first;    // first padded path index of this iteration
    unsigned long long next_path;    // next padded path index not yet generated
    unsigned long long total_paths;  // padded total
    unsigned long long rays;         // BVH queries so far
    unsigned long long paths;        // primary rays generated so far
    unsigned long long nodes_visited, prims_tested;
    unsigned long long iterations;
    unsigned long long cyc_generate, cyc_extend, cyc_shade;  // fused kernel: SM cycles per phase, summed over blocks
    uint32_t pad[2];
};

struct RenderConst {
    DCamera cam;
    RrsCamera cam64;  // the f64 camera, for the f64 sphere path (primary directions as lib.rs:202-210 computes them)
    uint32_t tiles_x, tiles_y;
    uint32_t small_index, magic_tiles, magic_tiles_y;  // division-free index math (primary_ray)
    uint32_t tiles, sblk_shift;   // tiles_x * tiles_y; log2 of the samples of one tile that are generated back to back
    uint32_t ws_shift;            // log2 of the width, in tiles, of the vertical stripes the tiles are walked in
    uint32_t exact_tiles;         // 1: the image is a whole number of 8x4 tiles (no padded lanes)
    unsigned long long npix_pad;  // tiles_x * tiles_y * 32
    uint32_t spp, sample_offset, max_bounces;
    uint64_t seed;
};

struct Wavefront {
    uint32_t capacity = 0;     // regions * region_cap
    uint32_t regions = 0;      // stripes == grid size of the persistent kernels
    uint32_t region_cap = 0;   // slots per stripe (multiple of 32)
    // both halves of the ping-pong in one allocation each: half k at offset k * capacity
    uint32_t* count = nullptr;  // [2][regions] rays per stripe
    float4* ray_o = nullptr;    // [2][capacity] origin xyz, origin primitive
    float4* ray_d = nullptr;    // [2][capacity] direction xyz, pixel
    float4* state = nullptr;    // [2][capacity] throughput rgb, sample << 8 | bounce
    float2* hits = nullptr;     // [capacity]    t, primitive
    double* org64 = nullptr;    // [2][capacity][3] f64 hit points of rays spawned on transmissive spheres
    float* wmis = nullptr;      // [2][capacity] MIS weight of continuation rays (RRS_FLAG_ENV_SAMPLING renders only)
    DCounters* counters = nullptr;
    DCounters* h_counters = nullptr;  // pinned
};

struct SceneImpl {
    int device = 0;
    int num_sms = 0;
    DScene d{};
    // owned device allocations
    char* geom_blob = nullptr;  // [nodes | primitives] in one allocation: one L2 access-policy window covers both
    size_t node_bytes = 0, geom_bytes = 0;
    size_t l2_persist_bytes = 0, l2_window_max = 0;  // 0: L2 persistence unavailable or switched off
    DPrim* prims = nullptr;     // into geom_blob
    DNode16* nodes = nullptr;   // into geom_blob
    DMat* mats = nullptr;
    float4* emis = nullptr;
    float4* hdri = nullptr;
    RrsPrim* prims_f64 = nullptr;
    RrsNodeF64* nodes_f64 = nullptr;
    double4* sphere64 = nullptr;
    double* tri64 = nullptr;
    // environment sampling table (env.cuh; env.wmis is set per render).  env_ok: the table exists, or the map is black
    // and there is nothing to sample (env.marg == nullptr); false when the map cannot be tabulated
    DEnv env{};
    bool env_ok = false;
    uint32_t n_prims = 0, n_nodes = 0;
    uint32_t max_depth = 0;
    double tmin = 0, tmax = 0;
    Wavefront wf;
    RrsStats stats{};
    float4* accum = nullptr;  // private accumulation buffer of rrs_render
    size_t accum_pixels = 0;
    unsigned long long* census = nullptr;  // [nan, negative]
    unsigned long long* h_census = nullptr;  // pinned
    float* resolve_dev = nullptr;     // device RGB image of rrs_render / rrs_resolve(host)
    float* resolve_pinned = nullptr;  // pinned staging for the device->host copy
    size_t resolve_bytes = 0;
    std::vector<cudaEvent_t> ev_pool;
    cudaStream_t own_stream = nullptr;  // rrs_render_multi without caller streams
    // rrs_render_accumulate is asynchronous: the statistics of the last render are completed by wf_finish_stats
    bool stats_pending = false;
    bool pending_split = false, pending_phases = false, pending_window = false;
    std::vector<size_t> phase_ev;  // event-pool indices of the per-iteration groups (RRS_FLAG_TIME_PHASES)
};

}  // namespace rrs

// the opaque handle of include/rayrs_b200.h
struct RrsScene {
    rrs::SceneImpl impl;
};

namespace rrs {

// wavefront.cu
int wf_render_accumulate(SceneImpl* s, const RrsCamera* cam, const RrsRenderParams* p, float4* d_accum,
                         cudaStream_t stream, std::string& err);
int wf_resolve(SceneImpl* s, const float4* d_accum, uint32_t w, uint32_t h, uint32_t spp_total, float* out,
               bool out_is_device, cudaStream_t stream, std::string& err);
int wf_to_raw_bytes(SceneImpl* s, const float4* d_accum, uint32_t w, uint32_t h, uint32_t spp_total, double gamma,
                    uint8_t* out, bool out_is_device, cudaStream_t stream, uint64_t* census3, std::string& err);
int wf_intersect32(SceneImpl* s, const RrsRay* rays, size_t n, int32_t* obj_id, double* t, std::string& err);
int wf_material_evaluate(SceneImpl* s, uint32_t material, const double* nv, const double* u, size_t n, float* out,
                         std::string& err);
int wf_background(SceneImpl* s, const double* dirs, size_t n, float* out, std::string& err);
int wf_rng_uniforms(SceneImpl* s, uint64_t seed, uint32_t pixel, uint32_t sample, uint32_t slot, float* out4,
                    std::string& err);
int wf_env_sample(SceneImpl* s, const double* u, size_t n, double* dir_pdf, std::string& err);
int wf_env_pdf(SceneImpl* s, const double* dirs, size_t n, double* pdf, std::string& err);
void wf_finish_stats(SceneImpl* s);  // waits for the last render of this scene and completes s->stats
void wf_free(SceneImpl* s);
// verify_f64.cu
int vf_intersect64(SceneImpl* s, const RrsRay* rays, size_t n, int32_t* obj_id, double* t, std::string& err);
// nee.cu
int nee_material_evaluate_pdf(SceneImpl* s, uint32_t material, const RrsPrim* light, const double* pnv, const double* u,
                              size_t n, double* out, std::string& err);

// Scratch device allocation of one entry point: freed on every return path, including the early returns of
// RRS_CUDA_CHECK.
template <typename T>
struct DevBuf {
    T* p = nullptr;
    DevBuf() = default;
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    ~DevBuf() { if (p) cudaFree(p); }
    cudaError_t alloc(size_t count) { return cudaMalloc(&p, sizeof(T) * (count ? count : 1)); }
    operator T*() const { return p; }
};

#define RRS_CUDA_CHECK(expr, errstr)                                                           \
    do {                                                                                       \
        cudaError_t _e = (expr);                                                               \
        if (_e != cudaSuccess) {                                                               \
            (errstr) = std::string(#expr) + ": " + cudaGetErrorString(_e);                     \
            return RRS_ERR_CUDA;                                                               \
        }                                                                                      \
    } while (0)

}  // namespace rrs
