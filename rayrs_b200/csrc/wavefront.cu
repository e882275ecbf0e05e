// Wavefront path tracer for sm_100a.  Replaces the pixel x spp x bounce loops of rayrs/src/main.rs:61-94 and
// rayrs-lib/src/lib.rs:521-560.
//
// A render is ONE launch of the persistent kernel k_wavefront.  Block b owns stripe b of the ray / state / hit
// queues in HBM and loops until the global path cursor is exhausted and its stripe has drained:
//   BVH form (k_wavefront<false,..>), per iteration of a block:
//     generate   Camera::generate_primary_ray (lib.rs:202-210) for new paths, appended behind the stripe's
//                survivors (path regeneration keeps the stripe full);
//     extend     closest hit per ray (intersect.cuh): warp-batched traversal of the flattened reference BVH with
//                dynamic ray fetch, traversal stacks in shared memory;
//     shade      Material::evaluate + emission + Russian roulette + background (shade_hit / shade_miss); survivors
//                are compacted into the other half of the stripe (__ballot_sync/__popc + one shared-memory
//                atomicAdd per warp); terminated paths add their radiance to the fp32 accumulator with one
//                128-bit reduction.
//   small-scene form (k_wavefront<true,..>, <= 8 primitives): one fused pass per iteration
//     (small_scene_iteration): survivors read from the queue, new paths generated in registers, closest hit by
//     brute force over the primitives staged in shared memory, shading, compaction.
// k_generate / k_extend / k_shade (+ k_plan) are the same phases as separate launches (RRS_FLAG_SPLIT_KERNELS, for
// per-phase profiling); k_pathloop is the register-resident alternative for small scenes (RRS_FLAG_FORCE_PATHLOOP).
#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdio>
#include <cstring>

#include "intersect.cuh"
#include "shading.cuh"
#include "wavefront.cuh"

namespace rrs {

#ifndef RRS_BLOCK_THREADS
#define RRS_BLOCK_THREADS 128
#endif
static constexpr int kBlock = RRS_BLOCK_THREADS;
// (The extend and shade phases as separate, not inlined device functions — so that the register allocation of one
// cannot cost the other spills — crash the compiler of this toolkit: nvcc 12.9 segfaults on the file.)
// The f64 distance of the accepted triangle hit (triangle_t64, intersect.cuh) is what rrs_intersect reports.  The
// render keeps the fp32 distance of the traversal: re-evaluating it in shade_hit would move the hit point by < 2e-6
// relative — far below what the image can see — and it cost configuration 5 (SPH64 form, 72 registers) 4.7 %
// (shade 17.6 -> 21.2 ms, profiles/ab_logs/ab_r02g_refine.log).  // threads per block of the persistent kernels
#ifndef RRS_BLOCKS_PER_SM
#define RRS_BLOCKS_PER_SM 8
#endif
#ifndef RRS_BLOCKS_PER_SM_F64
#define RRS_BLOCKS_PER_SM_F64 7
#endif

__device__ __forceinline__ uint32_t lane_id() { return threadIdx.x & 31u; }

// the persisting-L2 set-aside (cudaLimitPersistingL2CacheSize) as this library last set it, per device
static constexpr int kMaxDevices = 64;
static constexpr size_t kUnknownSetAside = ~(size_t)0;
static std::atomic<size_t> g_l2_set_aside[kMaxDevices];  // zero-initialised = the driver's default (no set-aside)

// Queue traffic streams (every ray / state / hit record is written once and read once): ld/st.global.cs marks the
// lines evict-first so that they do not push the BVH out of L2 (see "L2 residency" in wf_render_accumulate).
// Samples of one 8x4 pixel tile generated back to back (log2; see primary_ray).  Measured against sample-major order
// (profiles/ab_logs/ab_r02y_sample_block_*.log, ab_r02z_sample_block_large.log): 16 / 64 / 256 samples per block give
// configuration 4 +5.2 / +6.9 / +7.5 %, configuration 5 +3.6 / +4.0 / +4.3 %, the sphere series +1.5 … 3 %; 1024 is
// 1.6 % / 0.6 % behind 256 (too few tiles in flight: the float4 atomics of a pixel start to queue).
#ifndef RRS_SAMPLE_BLOCK_LOG2
#define RRS_SAMPLE_BLOCK_LOG2 8
#endif
// Width (log2, in 8x4 tiles) of the vertical stripes the tiles are walked in: 1 / 4 / 16 / 64 tiles wide give
// configuration 5 +0.7 / +0.9 / +1.0 / +0.9 % and configuration 4 +0.3 / +0.3 / +0.7 / +0.7 % over row-major order
// (profiles/ab_logs/ab_r03a_tile_stripes.log).
#ifndef RRS_TILE_STRIPE_LOG2
#define RRS_TILE_STRIPE_LOG2 4
#endif
#ifndef RRS_QUEUE_STREAMING
#define RRS_QUEUE_STREAMING 1
#endif
template <typename T>
__device__ __forceinline__ T ldq(const T* p) {
#if RRS_QUEUE_STREAMING
    return __ldcs(p);
#else
    return *p;
#endif
}
template <typename T>
__device__ __forceinline__ void stq(T* p, T v) {
#if RRS_QUEUE_STREAMING
    __stcs(p, v);
#else
    *p = v;
#endif
}

// ---------------------------------------------------------------------------------------
// Queue layout: the ray / state / hit queues are split into `regions` stripes of `region_cap`
// slots; block b of every kernel owns stripe b.  All queue bookkeeping (work cursor, append
// cursor of the compaction) is therefore a SHARED-MEMORY atomic; the only global atomics left
// are one per block per iteration (claiming new paths, ray statistics).  The first version of
// this file used one global work cursor and one global append counter: ncu showed 75 % of
// k_shade's stall samples on the shuffle behind those two same-address atomics
// (profiles/r01a_c2_globalqueue_stalls.txt).
// ---------------------------------------------------------------------------------------
// Both halves of the ping-pong live in ONE allocation per array (half k at offset k * capacity), so a
// kernel selects its half with one integer instead of a second set of pointers.
struct QueueSet {
    float4* ray_o;     // [2][capacity] origin xyz, origin primitive
    float4* ray_d;     // [2][capacity] direction xyz, pixel
    float4* state;     // [2][capacity] throughput rgb, sample << 8 | bounce
    float2* hits;      // [capacity]    t, primitive
    uint32_t* count;   // [2][regions]  rays per stripe
    double* org64;     // [2][capacity][3] f64 origins (transmissive spheres) or nullptr
    uint32_t capacity;  // regions * region_cap
    uint32_t regions;
    uint32_t region_cap;
};

// ---------------------------------------------------------------------------------------
// plan (1 thread): rotate the live-ray counters, raise `done`
// ---------------------------------------------------------------------------------------
__global__ void k_plan(DCounters* c) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    uint32_t live = c->n_next;
    c->n_cur = live;
    c->n_next = 0;
    c->done = (live == 0 && c->next_path >= c->total_paths) ? 1u : 0u;
    if (!c->done) c->iterations++;
}

// ---------------------------------------------------------------------------------------
// Camera::generate_primary_ray (lib.rs:202-210) for padded path index p.  Paths are numbered
// over 8x4 pixel tiles (one tile per 32 consecutive indices), so a warp that takes 32 consecutive indices starts
// coherent; a block of samples of one tile, then the next tile (see below).
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ bool primary_ray(const RenderConst& rc, unsigned long long p, uint32_t& pixel, uint32_t& sample,
                                            float3& d) {
    // path index -> (sample block, tile, sample within the block, lane): a warp is one 8x4 tile at one sample, the
    // 2^sblk_shift samples of a block follow each other, then the next tile; the next block starts after the last tile.
    // Tiles run row by row inside vertical stripes 2^ws_shift tiles wide, stripe after stripe: the ~1000 tiles in
    // flight are a compact patch of the image (128 x 256 pixels), not a line 8 pixels high across its whole width.
    // (Sample-major order — the whole image once per sample — keeps every pixel of a 4K image in flight at once: 133 MB
    // of accumulator lines visited by scattered float4 atomics, in an L2 the queues and the tree want; and the warps an
    // SM generates one after the other then start in different parts of the tree instead of on the same nodes.)
    // No 64-bit or 32-bit hardware division where the host could prove the multiply-high forms exact
    // (rc.small_index): p < 2^32.
    uint32_t s_local, tile, ty, stripe;
    const uint32_t l = (uint32_t)p & 31u;
    if (rc.small_index) {
        const uint32_t q = (uint32_t)p >> 5;
        const uint32_t q2 = q >> rc.sblk_shift;
        uint32_t s_blk = __umulhi(q2, rc.magic_tiles);
        tile = q2 - s_blk * rc.tiles;
        if (tile >= rc.tiles) {  // the magic quotient can be one short
            tile -= rc.tiles;
            ++s_blk;
        }
        s_local = (s_blk << rc.sblk_shift) | (q & ((1u << rc.sblk_shift) - 1u));
        const uint32_t a = tile >> rc.ws_shift;
        stripe = __umulhi(a, rc.magic_tiles_y);
        ty = a - stripe * rc.tiles_y;
        if (ty >= rc.tiles_y) {
            ty -= rc.tiles_y;
            ++stripe;
        }
    } else {
        const unsigned long long q = p >> 5;
        const unsigned long long q2 = q >> rc.sblk_shift;
        const uint32_t s_blk = (uint32_t)(q2 / rc.tiles);
        tile = (uint32_t)(q2 - (unsigned long long)s_blk * rc.tiles);
        s_local = (s_blk << rc.sblk_shift) | ((uint32_t)q & ((1u << rc.sblk_shift) - 1u));
        const uint32_t a = tile >> rc.ws_shift;
        stripe = a / rc.tiles_y;
        ty = a - stripe * rc.tiles_y;
    }
    const uint32_t tx = (stripe << rc.ws_shift) | (tile & ((1u << rc.ws_shift) - 1u));
    const uint32_t col = tx * 8u + (l & 7u);
    const uint32_t row = ty * 4u + (l >> 3);
    if (!rc.exact_tiles && !(col < rc.cam.W && row < rc.cam.H)) return false;  // padded tile lane outside the image
    pixel = row * rc.cam.W + col;
    sample = rc.sample_offset + s_local;
    float4 u = rng_uniforms(rc.seed, pixel, sample, 0u);
    // rayrs/src/main.rs:71-76: camera indices are (H - row, W - col)   (SURVEY.md F8)
    float fi = (float)(rc.cam.H - row), fj = (float)(rc.cam.W - col);
    float x = (fj + u.x) * rc.cam.inv_ppc - rc.cam.half_w;
    float y = (fi + u.y) * rc.cam.inv_ppc - rc.cam.half_h;
    d = add3(add3(rc.cam.z, scale3(rc.cam.e_x, x)), scale3(rc.cam.e_y, y));
    return true;
}

// ---------------------------------------------------------------------------------------
// generate: refill stripe b behind its survivors with new primary rays
// ---------------------------------------------------------------------------------------
// ENV (RRS_FLAG_ENV_SAMPLING): a path can have two rays in the next bounce (continuation + shadow ray), so the stripe
// is filled to half its capacity; rays already in it (paths and shadow rays) count against that half.
template <bool ENV = false>
__device__ __forceinline__ void phase_generate(const RenderConst& rc, DCounters* __restrict__ c, const QueueSet& q, int cur,
                                               uint32_t* s_u32, unsigned long long* s_u64) {
    const uint32_t b = blockIdx.x;
    uint32_t* __restrict__ count = q.count + (size_t)cur * q.regions;
    const uint32_t n0 = count[b];
    if (threadIdx.x == 0) {
        uint32_t need = ENV ? (q.region_cap / 2u > n0 ? q.region_cap / 2u - n0 : 0u) : q.region_cap - n0, got = 0;
        unsigned long long base = 0;
        // claim `need` consecutive padded path indices (one global atomic per block per iteration)
        if (need && c->next_path < c->total_paths) {
            base = atomicAdd(&c->next_path, (unsigned long long)need);
            if (base < c->total_paths) {
                unsigned long long left = c->total_paths - base;
                got = left < need ? (uint32_t)left : need;
            }
        }
        s_u64[0] = base;
        s_u32[0] = got;
        s_u32[1] = n0;  // append cursor
    }
    __syncthreads();
    const uint32_t got = s_u32[0];
    const unsigned long long first = s_u64[0];
    const uint32_t lane = lane_id();
    const size_t off = (size_t)cur * q.capacity + (size_t)b * q.region_cap;
    float4* __restrict__ ray_o = q.ray_o + off;
    float4* __restrict__ ray_d = q.ray_d + off;
    float4* __restrict__ state = q.state + off;
    const uint32_t got_pad = (got + 31u) & ~31u;
    for (uint32_t k = threadIdx.x; k < got_pad; k += blockDim.x) {
        bool valid = k < got;
        uint32_t pixel = 0, sample = 0;
        float3 d = f3(0.f, 0.f, 0.f);
        if (valid) valid = primary_ray(rc, first + k, pixel, sample, d);
        uint32_t slot;
        if (rc.exact_tiles) {  // warp-uniform
            slot = n0 + k;
        } else {
            uint32_t ballot = __ballot_sync(0xFFFFFFFFu, valid);
            uint32_t base = 0;
            if (lane == 0 && ballot) base = atomicAdd(&s_u32[1], __popc(ballot));
            base = __shfl_sync(0xFFFFFFFFu, base, 0);
            slot = base + __popc(ballot & ((1u << lane) - 1u));
        }
        if (!valid) continue;
        RRS_CHECK(slot < q.region_cap);
        stq(ray_o + slot, make_float4(rc.cam.origin.x, rc.cam.origin.y, rc.cam.origin.z, __uint_as_float(RRS_NO_PRIM)));
        stq(ray_d + slot, make_float4(d.x, d.y, d.z, __uint_as_float(pixel)));
        stq(state + slot, make_float4(1.f, 1.f, 1.f, __uint_as_float(sample << 8)));
    }
    __syncthreads();
    if (threadIdx.x == 0) count[b] = rc.exact_tiles ? n0 + got : s_u32[1];
}

__global__ void __launch_bounds__(kBlock) k_generate(RenderConst rc, DCounters* __restrict__ c, QueueSet q, int cur) {
    __shared__ uint32_t s_u32[2];
    __shared__ unsigned long long s_u64[1];
    phase_generate(rc, c, q, cur, s_u32, s_u64);
}

// ---------------------------------------------------------------------------------------
// extend: closest hit for every ray of stripe b; warps pull 32-ray batches from a shared cursor
// ---------------------------------------------------------------------------------------
// Warp-batched traversal with dynamic ray fetch.  The loop below is warp-uniform (every decision is
// a ballot), so the 32 lanes always execute the same kind of step:
//   refill   lanes without a ray take the next rays of the stripe as soon as `refill_lanes` of them are
//            idle — a ray that ends after 3 nodes no longer idles its lane while a neighbour walks 60
//            (the 32-rays-per-warp batch of the first version ran the node loop with 13.4 of 32 lanes
//            active on the 1M-triangle scene: profiles/r01c_c4_fused_metrics.csv);
//   nodes    inner-node steps while at least as many lanes want one as are parked on a leaf;
//   leaf     all parked lanes test their leaf run together, pop, and the cycle repeats.
template <bool COUNT>
__device__ __forceinline__ void flush_trav_counters(DCounters* __restrict__ c, const TravCounters& cnt) {
    if (COUNT) {
        uint32_t a = cnt.nodes, p = cnt.prims;
        for (int o = 16; o > 0; o >>= 1) {
            a += __shfl_xor_sync(0xFFFFFFFFu, a, o);
            p += __shfl_xor_sync(0xFFFFFFFFu, p, o);
        }
        if (lane_id() == 0) {
            atomicAdd(&c->nodes_visited, (unsigned long long)a);
            atomicAdd(&c->prims_tested, (unsigned long long)p);
        }
    }
}

template <bool BRUTE, bool COUNT, bool SPH64>
__device__ __forceinline__ void phase_extend(const DScene& sc, DCounters* __restrict__ c, const QueueSet& q, int cur,
                                             uint32_t* s_stack, const DPrim* s_prims, uint32_t* s_cursor) {
    const uint32_t FULL = 0xFFFFFFFFu;
    const uint32_t b = blockIdx.x;
    const uint32_t n = q.count[(size_t)cur * q.regions + b];
    const uint32_t lane = lane_id();
    const uint32_t lt_mask = (1u << lane) - 1u;
    const size_t roff = (size_t)b * q.region_cap, off = (size_t)cur * q.capacity + roff;
    const float4* __restrict__ ray_o = q.ray_o + off;
    const float4* __restrict__ ray_d = q.ray_d + off;
    float2* __restrict__ hits = q.hits + roff;
    if (BRUTE) {
        // small scene: every lane runs the same loop over the staged primitives, 32 rays per fetch
        TravCounters cnt{0, 0};
        for (;;) {
            uint32_t base = 0;
            if (lane == 0) base = atomicAdd(s_cursor, 32u);
            base = __shfl_sync(FULL, base, 0);
            if (base >= n) break;
            const uint32_t i = base + lane;
            if (i < n) {
                float4 o4 = ldq(ray_o + i), d4 = ldq(ray_d + i);
                const double* o64 = (SPH64 && q.org64) ? q.org64 + 3 * (off + i) : nullptr;
                float t;
                uint32_t prim;
                closest_hit_brute<COUNT, SPH64>(sc, s_prims, xyz(o4), xyz(d4), __float_as_uint(o4.w), o64, t, prim, cnt);
                stq(hits + i, make_float2(t, __uint_as_float(prim)));
            }
        }
        flush_trav_counters<COUNT>(c, cnt);
        return;
    }
    // inner-node steps a lane takes per ballot round (round 1 swept 1..8: 3-4 best, profiles/ab_logs/sweep_tune*.log;
    // round 2, after the register diet: 2 / 3 / 4 / 6 within +-0.5 %, ab_r02n_sweep.log)
    constexpr uint32_t kNodeSteps = 4;
    // the node rounds go on while want * RRS_LEAF_NUM >= parked * RRS_LEAF_DEN lanes ask for one (1 / 1: as many lanes on
    // inner nodes as are parked on a leaf); 2 / 1 = leaves later with fuller warps, 1 / 2 = leaves sooner — measurement switch
#ifndef RRS_LEAF_NUM
#define RRS_LEAF_NUM 1
#define RRS_LEAF_DEN 1
#endif
    SStack stack;
    stack.init(s_stack + threadIdx.x, blockDim.x);
    TravCounters cnt{0, 0};
    RayK r;
    Trav tv;
    tv.cur = TRAV_DONE;
    tv.sp = 1;
    tv.tbest = 0.f;
    tv.best = RRS_NO_PRIM;
    bool exhausted = false;
    constexpr uint32_t kNoRay = 0xFFFFFFFFu;
    uint32_t my_i = kNoRay;  // queue slot of the lane's ray; kNoRay while the lane is idle
    for (;;) {
        // ---- refill ----
        uint32_t idle = __ballot_sync(FULL, my_i == kNoRay);
        if (!exhausted && (uint32_t)__popc(idle) >= sc.refill_lanes) {
            uint32_t base = 0;
            if (lane == 0) base = atomicAdd(s_cursor, (uint32_t)__popc(idle));
            base = __shfl_sync(FULL, base, 0);
            exhausted = base + (uint32_t)__popc(idle) >= n;
            const uint32_t i = base + (uint32_t)__popc(idle & lt_mask);
            if (my_i == kNoRay && i < n) {
                float4 o4 = ldq(ray_o + i), d4 = ldq(ray_d + i);
                trav_begin(sc, xyz(o4), xyz(d4), __float_as_uint(o4.w), stack, r, tv);
                my_i = i;
            }
            idle = __ballot_sync(FULL, my_i == kNoRay);
        }
        if (idle == FULL) {
            if (exhausted) break;
            continue;  // fewer idle lanes than the threshold cannot be all 32: unreachable, kept for safety
        }
        // ---- inner nodes ----
        for (;;) {
            const bool inner = trav_on_inner(tv);
            const uint32_t want = __ballot_sync(FULL, inner);
            const uint32_t parked = __ballot_sync(FULL, !inner && tv.cur != TRAV_DONE);
            if (want == 0u || __popc(want) * RRS_LEAF_NUM < __popc(parked) * RRS_LEAF_DEN) break;
            if (inner) {
                trav_node_step<COUNT>(sc, r, tv, stack, cnt);
#pragma unroll 1
                for (uint32_t k = 1; k < kNodeSteps && trav_on_inner(tv); ++k) trav_node_step<COUNT>(sc, r, tv, stack, cnt);
            }
        }
        // ---- leaves ----
        if (!trav_on_inner(tv) && tv.cur != TRAV_DONE)
            trav_leaf_step<COUNT, SPH64>(sc, r, tv, stack, (SPH64 && q.org64) ? q.org64 + 3 * (off + my_i) : nullptr, cnt);
        if (my_i != kNoRay && tv.cur == TRAV_DONE) {  // finished (in a node step or in the leaf step)
            stq(hits + my_i, make_float2(tv.tbest, __uint_as_float(tv.best)));
            my_i = kNoRay;
        }
    }
    flush_trav_counters<COUNT>(c, cnt);
}

template <bool BRUTE, bool COUNT, bool SPH64>
__global__ void __launch_bounds__(kBlock) k_extend(DScene sc, DCounters* __restrict__ c, QueueSet q, int cur) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    // [stack_entries * blockDim.x * 4 B traversal stacks]
    uint32_t* s_stack = reinterpret_cast<uint32_t*>(smem_raw);
    __shared__ DPrim s_prims[RRS_BRUTE_MAX];
    __shared__ uint32_t s_cursor;
    if (threadIdx.x == 0) s_cursor = 0;
    stage_brute_prims(sc, s_prims);
    __syncthreads();
    phase_extend<BRUTE, COUNT, SPH64>(sc, c, q, cur, s_stack, s_prims, &s_cursor);
}

// ---------------------------------------------------------------------------------------
// One path vertex: Material::evaluate + emission + Russian roulette (lib.rs:532-551) for a ray that hit
// `prim` at distance t.  Shared by the queue-based shade phase and the register-resident path loop.
// ---------------------------------------------------------------------------------------
// Sphere::intersect, Ray::point, Sphere::normal in the reference's f64 arithmetic for a hit on a transmissive sphere
// (intersect.cuh, "sphere re-entry").  (Kept out of line — __noinline__, so that its f64 temporaries would not count
// against every path's registers — it costs config 3 31 % and config 5 5 %: the call's register save / restore and the
// hit point passed through local memory outweigh the spills it removes; profiles/ab_logs/ab_r02r_outline.log.)
__device__ __forceinline__ void sphere_hit_point64(const DScene& sc, const RenderConst& rc, uint32_t pixel, uint32_t sample, float4 o4, float4 d4,
                                    float t32, uint32_t sphere_index, const double* o64_in, double* p64, float3* pos, float3* nrm) {
    const uint32_t ow = __float_as_uint(o4.w);
    double ox = o4.x, oy = o4.y, oz = o4.z;
    if (ow != RRS_NO_PRIM && (ow & RRS_ORG64) && o64_in) {
        ox = o64_in[0]; oy = o64_in[1]; oz = o64_in[2];
    }
    double dx = d4.x, dy = d4.y, dz = d4.z;
    if (ow == RRS_NO_PRIM) {
        // primary ray: Camera::generate_primary_ray (lib.rs:202-210) in f64.  The loss
        // probability of the re-entry quirk depends on the f64 rounding of the FIRST hit,
        // and an fp32-exact direction makes that arithmetic atypically exact (measured:
        // 81 % instead of 71 % for the outer spheres), so the direction is rebuilt here.
        const RrsCamera& c64 = rc.cam64;
        uint32_t row = pixel / rc.cam.W, col = pixel - row * rc.cam.W;
        float4 u0 = rng_uniforms(rc.seed, pixel, sample, 0u);
        double fj = (double)(rc.cam.W - col), fi = (double)(rc.cam.H - row), ppc = (double)c64.ppc;
        double x = __dsub_rn(__ddiv_rn(__dadd_rn(fj, (double)u0.x), ppc), __ddiv_rn(c64.width, 2.));
        double y = __dsub_rn(__ddiv_rn(__dadd_rn(fi, (double)u0.y), ppc), __ddiv_rn(c64.height, 2.));
        dx = __dadd_rn(__dadd_rn(c64.z_scaled[0], __dmul_rn(x, c64.e_x[0])), __dmul_rn(y, c64.e_y[0]));
        dy = __dadd_rn(__dadd_rn(c64.z_scaled[1], __dmul_rn(x, c64.e_x[1])), __dmul_rn(y, c64.e_y[1]));
        dz = __dadd_rn(__dadd_rn(c64.z_scaled[2], __dmul_rn(x, c64.e_x[2])), __dmul_rn(y, c64.e_y[2]));
        ox = c64.origin[0]; oy = c64.origin[1]; oz = c64.origin[2];
    }
    const double4 s64 = sc.sphere64[sphere_index];
    double t64;
    const bool ok = sphere_intersect64(s64, ox, oy, oz, dx, dy, dz, t64);
    if (!ok || fabs(t64 - (double)t32) > 1e-3 * (double)t32) t64 = (double)t32;  // rim: keep the fp32 root
    const double px = __dadd_rn(ox, __dmul_rn(dx, t64)), py = __dadd_rn(oy, __dmul_rn(dy, t64)), pz = __dadd_rn(oz, __dmul_rn(dz, t64));
    p64[0] = px; p64[1] = py; p64[2] = pz;
    const double nx = __dsub_rn(px, s64.x), ny = __dsub_rn(py, s64.y), nz = __dsub_rn(pz, s64.z);
    // Sphere::normal (geometry.rs:134-136) is only ever consumed in fp32 here: scale by 1/r in f64 (one multiply
    // per component; |p - c| = r to 1e-16) so the fp32 normalisation below starts from O(1) components
    const double inv_r = (double)rsqrtf((float)s64.w);
    *nrm = normalize3(f3((float)(nx * inv_r), (float)(ny * inv_r), (float)(nz * inv_r)));
    *pos = f3((float)px, (float)py, (float)pz);
}

struct NextRay {
    bool alive, carry64;
    float4 no, nd, ns;           // origin + origin word, direction + pixel, throughput + (sample << 8 | bounce)
    double p64[3];               // f64 hit point (transmissive spheres; written only when carry64)
};

// ENV: next-event estimation of the environment at a Lambertian or Cook-Torrance vertex (env.cuh).  *shadow gets the
// shadow ray (its state carries what it adds if it escapes), *wcont the MIS weight of the continuation ray's escape.
template <bool SPH64, bool STAGED, bool ENV = false>
__device__ __forceinline__ NextRay shade_hit(const DScene& sc, const RenderConst& rc, float4* __restrict__ accum, float2 h,
                                             float4 o4, float4 d4, float4 st, const double* o64_in,
                                             const DEnv* env = nullptr, NextRay* shadow = nullptr, float* wcont = nullptr) {
    NextRay nr;
    nr.alive = false;
    nr.carry64 = false;
    bool& alive = nr.alive;
    bool& carry64 = nr.carry64;
    float4 &no = nr.no, &nd = nr.nd, &ns = nr.ns;
    uint32_t prim = __float_as_uint(h.y);
    uint32_t pixel = __float_as_uint(d4.w);
    RRS_CHECK(prim < sc.n_prims && pixel < rc.cam.W * rc.cam.H);
    uint32_t sb = __float_as_uint(st.w);
    uint32_t bounce = sb & 0xFFu, sample = sb >> 8;
    float3 thr = xyz(st);
    float3 o = xyz(o4), d = xyz(d4);
    const float4* pp = reinterpret_cast<const float4*>(sc.prims + prim);
    float4 a = __ldg(pp);
    const float4* mp = reinterpret_cast<const float4*>(sc.mats + prim_material(a));
    DMat m;
    m.m0 = __ldg(mp);
    float3 pos, nrm;
    const uint32_t mtag = __float_as_uint(m.m0.w);
    const bool transmissive = mtag == RRS_MAT_REFRACT || mtag == RRS_MAT_GLASS ||
                              mtag == RRS_MAT_COOK_TORRANCE_REFRACT || mtag == RRS_MAT_COOK_TORRANCE_GLASS;
    if (SPH64 && sc.sphere64 != nullptr && prim_type(a) == RRS_SPHERE && transmissive) {
        // hit point on a transmissive sphere in the reference's f64 arithmetic
        sphere_hit_point64(sc, rc, pixel, sample, o4, d4, h.x, __float_as_uint(__ldg(pp + 1).y), o64_in, nr.p64, &pos, &nrm);
        carry64 = true;
    } else {
        pos = madd3(d, h.x, o);  // Ray::point lib.rs:41-43
        nrm = prim_normal(sc.prims, prim, a, pos);
    }
    float3 view = normalize3(neg3(d));
    float4 u = rng_uniforms(rc.seed, pixel, sample, bounce + 1u);
    m.m1 = __ldg(mp + 1);
    m.m2 = __ldg(mp + 2);
    ScatterOut so = material_evaluate<STAGED>(m, nrm, view, u.x, u.y, u.z);
    // NEE applies where the plain render traces a continuation at all, and not to a delta lobe (alpha^2 == 0 in fp32)
    const bool nee = ENV && env->marg != nullptr && bounce + 1u < rc.max_bounces &&
                     (mtag == RRS_MAT_LAMBERTIAN || (mtag == RRS_MAT_COOK_TORRANCE && m.m1.w > 0.f));
    if (ENV) {
        shadow->alive = false;
        *wcont = 1.f;
    }
    if (nee) {
        const float4 ue = rng_uniforms(rc.seed, pixel, sample, RRS_ENV_SLOT + bounce);
        float3 l;
        const float pe = env_sample(sc, *env, ue.x, ue.y, ue.z, ue.w, l);
        float3 W;
        const float pb = pe > 0.f ? nee_bsdf(m, mtag, nrm, view, l, W) : 0.f;
        const float3 tw = mul3(thr, W);
        const float p = fmaxf(fmaxf(tw.x, tw.y), tw.z);
        if (pb > 0.f && p > 0.f) {
            // the plain continuation survives Russian roulette with min(p, 1) and is divided by p
            const float k = fminf(p, 1.f) / p * mis_cross(pe, pb);
            const float3 bg = background(sc, l);
            shadow->alive = true;
            shadow->no = make_float4(pos.x, pos.y, pos.z, __uint_as_float(prim | RRS_SHADOW));
            shadow->nd = make_float4(l.x, l.y, l.z, d4.w);
            shadow->ns = make_float4(tw.x * bg.x * k, tw.y * bg.y * k, tw.z * bg.z * k, __uint_as_float(sb));
        }
    }
    bool finished = true;
    if (so.scatter) {
        // lib.rs:533-547
        int emi = __float_as_int(__ldg(pp + 2).w);
        if (emi >= 0) {
            float4 e = __ldg(sc.emis + emi);
            atomicAdd(accum + pixel, make_float4(thr.x * e.x, thr.y * e.y, thr.z * e.z, 0.f));
        }
        thr = mul3(thr, so.color);
        float p = fmaxf(fmaxf(thr.x, thr.y), thr.z);
        // lib.rs:543-546: `if random() > p { break }`, then thr / p.  p == 0 (a black surface) ends the path here: the
        // 24-bit uniform is exactly 0 once in 2^24 draws, and surviving on it would put 0/0 into the accumulator
        if (p > 0.f && !(u.w > p) && bounce + 1u < rc.max_bounces) {
            thr = f3(thr.x / p, thr.y / p, thr.z / p);
            finished = false;
            alive = true;
            no = make_float4(pos.x, pos.y, pos.z, __uint_as_float(carry64 ? (prim | RRS_ORG64) : prim));
            nd = make_float4(so.dir.x, so.dir.y, so.dir.z, d4.w);
            ns = make_float4(thr.x, thr.y, thr.z, __uint_as_float((sample << 8) | (bounce + 1u)));
            if (nee) {
                float3 W;
                const float pb = nee_bsdf(m, mtag, nrm, view, so.dir, W);
                const float pe = env_pdf(sc, *env, so.dir);
                *wcont = pe > 0.f ? mis_power(pb, pe) : 1.f;
            }
        }
    }
    if (finished) atomicAdd(accum + pixel, make_float4(0.f, 0.f, 0.f, 1.f));
    return nr;
}

// lib.rs:552-556: light + throughput * background(direction)
__device__ __forceinline__ void shade_miss(const DScene& sc, float4* __restrict__ accum, float4 d4, float4 st) {
    float3 bg = background(sc, xyz(d4));
    atomicAdd(accum + __float_as_uint(d4.w), make_float4(st.x * bg.x, st.y * bg.y, st.z * bg.z, 1.f));
}

// ---------------------------------------------------------------------------------------
// shade: Material::evaluate + Russian roulette + background for stripe b of queue `cur`;
// survivors are compacted into stripe b of the other queue
// ---------------------------------------------------------------------------------------
// INLINE_HIT (small scenes in the queued kernel): the closest hit is found here, by brute force over the staged
// primitives, instead of in a separate extend phase — a fixed 8-primitive loop has nothing to gain from being
// batched on its own, and fusing it drops the hit queue and the second read of every ray record (48 of ~190 bytes
// of DRAM traffic per ray on the frosted-glass series, profiles/r01j_c3_frosted_metrics.csv).
// ENV (RRS_FLAG_ENV_SAMPLING): a shadow ray adds its state if it escapes and is dropped if it hits; a continuation
// ray's escape is weighted by its MIS weight (env_miss); a shaded vertex may emit a shadow ray besides its
// continuation (env_compact).
__device__ __forceinline__ void env_miss(const DScene& sc, const DEnv& env, float4* __restrict__ accum, float4 o4, float4 d4,
                                         float4 st, size_t slot) {
    const uint32_t ow = __float_as_uint(o4.w);
    if (ow != RRS_NO_PRIM && (ow & RRS_SHADOW)) {
        atomicAdd(accum + __float_as_uint(d4.w), make_float4(st.x, st.y, st.z, 0.f));  // not a path end: .w stays
        return;
    }
    const float w = ow == RRS_NO_PRIM ? 1.f : env.wmis[slot];  // camera rays: no other strategy
    shade_miss(sc, accum, d4, make_float4(st.x * w, st.y * w, st.z * w, st.w));
}

__device__ __forceinline__ bool is_shadow_ray(float4 o4) {
    const uint32_t ow = __float_as_uint(o4.w);
    return ow != RRS_NO_PRIM && (ow & RRS_SHADOW);
}

// survivors and shadow rays of this warp take consecutive slots of the stripe (survivors first)
template <bool SPH64>
__device__ __forceinline__ void env_compact(const QueueSet& q, const DEnv& env, size_t ooff, uint32_t* s_out, const NextRay& nr,
                                            const NextRay& sr, float wcont) {
    const uint32_t lane = lane_id(), lt = (1u << lane) - 1u;
    const uint32_t ba = __ballot_sync(0xFFFFFFFFu, nr.alive), bs = __ballot_sync(0xFFFFFFFFu, sr.alive);
    if ((ba | bs) == 0u) return;
    uint32_t obase = 0;
    if (lane == 0) obase = atomicAdd(s_out, __popc(ba) + __popc(bs));
    obase = __shfl_sync(0xFFFFFFFFu, obase, 0);
    if (nr.alive) {
        const uint32_t slot = obase + __popc(ba & lt);
        RRS_CHECK(slot < q.region_cap);
        stq(q.ray_o + ooff + slot, nr.no);
        stq(q.ray_d + ooff + slot, nr.nd);
        stq(q.state + ooff + slot, nr.ns);
        stq(env.wmis + ooff + slot, wcont);
        if (SPH64 && nr.carry64 && q.org64) {
            double* o64 = q.org64 + 3 * (ooff + slot);
            o64[0] = nr.p64[0]; o64[1] = nr.p64[1]; o64[2] = nr.p64[2];
        }
    }
    if (sr.alive) {
        const uint32_t slot = obase + __popc(ba) + __popc(bs & lt);
        RRS_CHECK(slot < q.region_cap);
        stq(q.ray_o + ooff + slot, sr.no);
        stq(q.ray_d + ooff + slot, sr.nd);
        stq(q.state + ooff + slot, sr.ns);
    }
}

template <bool SPH64, bool INLINE_HIT, bool COUNT, bool ENV = false>
__device__ __forceinline__ void phase_shade(const DScene& sc, const RenderConst& rc, DCounters* __restrict__ c,
                                            const QueueSet& q, int cur, float4* __restrict__ accum, uint32_t* s_cursor,
                                            uint32_t* s_out, const DPrim* s_prims, const DEnv* env = nullptr) {
    const uint32_t b = blockIdx.x;
    const uint32_t n = q.count[(size_t)cur * q.regions + b];
    const uint32_t lane = lane_id();
    const size_t roff = (size_t)b * q.region_cap;
    const size_t off = (size_t)cur * q.capacity + roff, ooff = (size_t)(cur ^ 1) * q.capacity + roff;
    const float4* __restrict__ ray_o = q.ray_o + off;
    const float4* __restrict__ ray_d = q.ray_d + off;
    const float4* __restrict__ state = q.state + off;
    const float2* __restrict__ hits = q.hits + roff;
    float4* __restrict__ out_o = q.ray_o + ooff;
    float4* __restrict__ out_d = q.ray_d + ooff;
    float4* __restrict__ out_state = q.state + ooff;
    TravCounters tcnt{0, 0};
    for (;;) {
        uint32_t base = 0;
        if (lane == 0) base = atomicAdd(s_cursor, 32u);
        base = __shfl_sync(0xFFFFFFFFu, base, 0);
        if (base >= n) break;
        uint32_t i = base + lane;
        NextRay nr;
        nr.alive = false;
        nr.carry64 = false;
        NextRay sr;
        sr.alive = false;
        float wcont = 1.f;
        if (i < n) {
            float4 o4 = ldq(ray_o + i), d4 = ldq(ray_d + i), st = ldq(state + i);
            const double* o64 = (SPH64 && q.org64) ? q.org64 + 3 * (off + i) : nullptr;
            float2 h;
            if (INLINE_HIT) {
                uint32_t prim;
                closest_hit_brute<COUNT, SPH64>(sc, s_prims, xyz(o4), xyz(d4), __float_as_uint(o4.w), o64, h.x, prim, tcnt);
                h.y = __uint_as_float(prim);
            } else {
                h = ldq(hits + i);
            }
            if (ENV) {
                if (__float_as_uint(h.y) == RRS_NO_PRIM) env_miss(sc, *env, accum, o4, d4, st, off + i);
                else if (!is_shadow_ray(o4)) nr = shade_hit<SPH64, true, true>(sc, rc, accum, h, o4, d4, st, o64, env, &sr, &wcont);
            } else if (__float_as_uint(h.y) == RRS_NO_PRIM) {
                shade_miss(sc, accum, d4, st);
            } else {
                nr = shade_hit<SPH64, true>(sc, rc, accum, h, o4, d4, st, o64);
            }
        }
        if (ENV) {
            env_compact<SPH64>(q, *env, ooff, s_out, nr, sr, wcont);
            continue;
        }
        const bool alive = nr.alive;
        // queue compaction: survivors of this warp take consecutive slots of the stripe
        uint32_t ballot = __ballot_sync(0xFFFFFFFFu, alive);
        if (ballot) {
            uint32_t obase = 0;
            if (lane == 0) obase = atomicAdd(s_out, __popc(ballot));
            obase = __shfl_sync(0xFFFFFFFFu, obase, 0);
            if (alive) {
                uint32_t slot = obase + __popc(ballot & ((1u << lane) - 1u));
                RRS_CHECK(slot < q.region_cap);
                stq(out_o + slot, nr.no);
                stq(out_d + slot, nr.nd);
                stq(out_state + slot, nr.ns);
                if (SPH64 && nr.carry64 && q.org64) {
                    double* o64 = q.org64 + 3 * (ooff + slot);
                    o64[0] = nr.p64[0]; o64[1] = nr.p64[1]; o64[2] = nr.p64[2];
                }
            }
        }
    }
    if (INLINE_HIT) flush_trav_counters<COUNT>(c, tcnt);
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t survivors = *s_out;
        q.count[(size_t)(cur ^ 1) * q.regions + b] = survivors;
        if (n) atomicAdd(&c->rays, (unsigned long long)n);
        if (survivors) atomicAdd(&c->n_next, survivors);
    }
}

template <bool SPH64>
__global__ void __launch_bounds__(kBlock, SPH64 ? RRS_BLOCKS_PER_SM_F64 : RRS_BLOCKS_PER_SM) k_shade(DScene sc, RenderConst rc, DCounters* __restrict__ c,
                                                                  QueueSet q, int cur, float4* __restrict__ accum) {
    __shared__ uint32_t s_cursor, s_out;
    if (threadIdx.x == 0) {
        s_cursor = 0;
        s_out = 0;
    }
    __syncthreads();
    phase_shade<SPH64, false, false>(sc, rc, c, q, cur, accum, &s_cursor, &s_out, nullptr);
}

// ---------------------------------------------------------------------------------------
// Small scenes (BRUTE): one pass per iteration.  The stripe's survivors are read from the queue; the slots behind
// them are filled with NEW paths generated in registers (no queue write + read-back for primary rays); every ray
// finds its closest hit by brute force over the staged primitives, is shaded, and only the survivors of this
// bounce are written — compacted — into the other half of the stripe.  Per ray that leaves one 48-byte queue
// write and one 48-byte read for the ~36 % of rays that continue, instead of generate-write / extend-read /
// hit-write / shade-read (192 B of DRAM traffic per ray on the frosted-glass series, profiles/r01j_c3_frosted_*).
// ---------------------------------------------------------------------------------------
template <bool COUNT, bool SPH64, bool ENV = false>
__device__ __forceinline__ bool small_scene_iteration(const DScene& sc, const RenderConst& rc, DCounters* __restrict__ c,
                                                      const QueueSet& q, int cur, float4* __restrict__ accum,
                                                      const DPrim* s_prims, uint32_t* s_u32, unsigned long long* s_u64,
                                                      const DEnv* env = nullptr) {
    // s_u32: [0] new paths claimed, [1] rays traced, [2] work cursor, [3] append cursor; s_u64[0]: first new path index
    const uint32_t FULL = 0xFFFFFFFFu;
    const uint32_t b = blockIdx.x;
    const uint32_t lane = lane_id();
    const uint32_t lt_mask = (1u << lane) - 1u;
    const uint32_t n0 = q.count[(size_t)cur * q.regions + b];
    if (threadIdx.x == 0) {
        // ENV: fill to half the stripe, as phase_generate does
        uint32_t need = ENV ? (q.region_cap / 2u > n0 ? q.region_cap / 2u - n0 : 0u) : q.region_cap - n0, got = 0;
        unsigned long long base = 0;
        if (need && c->next_path < c->total_paths) {  // one global atomic per block per iteration
            base = atomicAdd(&c->next_path, (unsigned long long)need);
            if (base < c->total_paths) {
                unsigned long long left = c->total_paths - base;
                got = left < need ? (uint32_t)left : need;
            }
        }
        s_u64[0] = base;
        s_u32[0] = got;
        s_u32[1] = 0;
        s_u32[2] = 0;
        s_u32[3] = 0;
    }
    __syncthreads();
    const uint32_t n = n0 + s_u32[0];
    const unsigned long long first = s_u64[0];
    if (n == 0) return false;  // nothing live and no path left for this block
    const size_t roff = (size_t)b * q.region_cap;
    const size_t off = (size_t)cur * q.capacity + roff, ooff = (size_t)(cur ^ 1) * q.capacity + roff;
    const float4* __restrict__ ray_o = q.ray_o + off;
    const float4* __restrict__ ray_d = q.ray_d + off;
    const float4* __restrict__ state = q.state + off;
    float4* __restrict__ out_o = q.ray_o + ooff;
    float4* __restrict__ out_d = q.ray_d + ooff;
    float4* __restrict__ out_state = q.state + ooff;
    TravCounters tcnt{0, 0};
    uint32_t traced = 0;
    for (;;) {
        uint32_t base = 0;
        if (lane == 0) base = atomicAdd(&s_u32[2], 32u);
        base = __shfl_sync(FULL, base, 0);
        if (base >= n) break;
        const uint32_t i = base + lane;
        NextRay nr;
        nr.alive = false;
        nr.carry64 = false;
        bool valid = i < n;
        float4 o4, d4, st;
        const double* o64 = nullptr;
        if (valid) {
            if (i < n0) {  // a survivor of the previous bounce
                o4 = ldq(ray_o + i);
                d4 = ldq(ray_d + i);
                st = ldq(state + i);
                if (SPH64 && q.org64) o64 = q.org64 + 3 * (off + i);
            } else {       // a new path: Camera::generate_primary_ray, straight into registers
                uint32_t pixel = 0, sample = 0;
                float3 d;
                valid = primary_ray(rc, first + (i - n0), pixel, sample, d);
                o4 = make_float4(rc.cam.origin.x, rc.cam.origin.y, rc.cam.origin.z, __uint_as_float(RRS_NO_PRIM));
                d4 = make_float4(d.x, d.y, d.z, __uint_as_float(pixel));
                st = make_float4(1.f, 1.f, 1.f, __uint_as_float(sample << 8));
            }
        }
        NextRay sr;
        sr.alive = false;
        float wcont = 1.f;
        if (valid) {
            float2 h;
            uint32_t prim;
            closest_hit_brute<COUNT, SPH64>(sc, s_prims, xyz(o4), xyz(d4), __float_as_uint(o4.w), o64, h.x, prim, tcnt);
            h.y = __uint_as_float(prim);
            ++traced;
            if (ENV) {
                if (prim == RRS_NO_PRIM) env_miss(sc, *env, accum, o4, d4, st, off + i);  // (new paths: camera rays)
                else if (!is_shadow_ray(o4)) nr = shade_hit<SPH64, true, true>(sc, rc, accum, h, o4, d4, st, o64, env, &sr, &wcont);
            } else if (prim == RRS_NO_PRIM) {
                shade_miss(sc, accum, d4, st);
            } else {
                nr = shade_hit<SPH64, true>(sc, rc, accum, h, o4, d4, st, o64);
            }
        }
        if (ENV) {
            env_compact<SPH64>(q, *env, ooff, &s_u32[3], nr, sr, wcont);
            continue;
        }
        // queue compaction: survivors of this warp take consecutive slots of the stripe's other half
        const uint32_t ballot = __ballot_sync(FULL, nr.alive);
        if (ballot) {
            uint32_t obase = 0;
            if (lane == 0) obase = atomicAdd(&s_u32[3], (uint32_t)__popc(ballot));
            obase = __shfl_sync(FULL, obase, 0);
            if (nr.alive) {
                const uint32_t slot = obase + __popc(ballot & lt_mask);
                RRS_CHECK(slot < q.region_cap);
                stq(out_o + slot, nr.no);
                stq(out_d + slot, nr.nd);
                stq(out_state + slot, nr.ns);
                if (SPH64 && nr.carry64 && q.org64) {
                    double* w64 = q.org64 + 3 * (ooff + slot);
                    w64[0] = nr.p64[0]; w64[1] = nr.p64[1]; w64[2] = nr.p64[2];
                }
            }
        }
    }
    for (int o = 16; o > 0; o >>= 1) traced += __shfl_xor_sync(FULL, traced, o);
    if (lane == 0 && traced) atomicAdd(&s_u32[1], traced);
    flush_trav_counters<COUNT>(c, tcnt);
    __syncthreads();
    if (threadIdx.x == 0) {
        const uint32_t survivors = s_u32[3];
        q.count[(size_t)(cur ^ 1) * q.regions + b] = survivors;
        if (s_u32[1]) atomicAdd(&c->rays, (unsigned long long)s_u32[1]);
        s_u64[4] += 1;
    }
    __syncthreads();
    return true;
}

// ---------------------------------------------------------------------------------------
// fused persistent kernel: because block b only ever touches stripe b, the three phases need no
// grid-wide ordering at all — every block runs its OWN generate -> extend -> shade loop until the
// global path cursor is exhausted and its stripe has drained.  One launch per render: no launch
// gaps, no per-kernel tails, no host polling; a stripe that was just written by shade is re-read
// by the same SM while it is still in L2.  The three-kernel form above is kept (RRS_FLAG_SPLIT_KERNELS)
// because it gives per-phase ncu evidence.
// ---------------------------------------------------------------------------------------
template <bool BRUTE, bool COUNT, bool SPH64, bool ENV>
__device__ __forceinline__ bool wavefront_iteration(const DScene& sc, const RenderConst& rc, DCounters* __restrict__ c,
                                                    const QueueSet& q, int cur, float4* __restrict__ accum,
                                                    uint32_t* s_stack, const DPrim* s_prims, uint32_t* s_u32,
                                                    unsigned long long* s_u64, const DEnv* env) {
    // s_u64[1..3]: cycles spent in generate / extend / shade, s_u64[4]: iterations (thread 0 only)
    long long t0 = 0;
    if (threadIdx.x == 0) t0 = clock64();
    phase_generate<ENV>(rc, c, q, cur, s_u32, s_u64);
    __syncthreads();
    const uint32_t n = q.count[(size_t)cur * q.regions + blockIdx.x];
    if (threadIdx.x == 0) {
        s_u32[2] = 0;  // work cursor
        s_u32[3] = 0;  // append cursor of the compaction
        long long t1 = clock64();
        s_u64[1] += (unsigned long long)(t1 - t0);
        t0 = t1;
    }
    __syncthreads();
    if (n == 0) return false;  // nothing live and no path left for this block
    if (!BRUTE) {
        phase_extend<BRUTE, COUNT, SPH64>(sc, c, q, cur, s_stack, s_prims, &s_u32[2]);
        __syncthreads();
        if (threadIdx.x == 0) {
            s_u32[2] = 0;
            long long t1 = clock64();
            s_u64[2] += (unsigned long long)(t1 - t0);
            t0 = t1;
        }
        __syncthreads();
    }
    phase_shade<SPH64, BRUTE, COUNT, ENV>(sc, rc, c, q, cur, accum, &s_u32[2], &s_u32[3], s_prims, env);
    __syncthreads();
    if (threadIdx.x == 0) {
        s_u64[3] += (unsigned long long)(clock64() - t0);
        s_u64[4] += 1;
    }
    return true;
}

template <bool BRUTE, bool COUNT, bool SPH64, bool ENV>
__device__ __forceinline__ void wavefront_kernel(const DScene& sc, const RenderConst& rc, DCounters* __restrict__ c,
                                                 const QueueSet& q, float4* __restrict__ accum, const DEnv* env) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    uint32_t* s_stack = reinterpret_cast<uint32_t*>(smem_raw);
    __shared__ DPrim s_prims[RRS_BRUTE_MAX];
    __shared__ uint32_t s_u32[4];
    __shared__ unsigned long long s_u64[5];
    if (threadIdx.x < 5) s_u64[threadIdx.x] = 0;
    stage_brute_prims(sc, s_prims);
    __syncthreads();
    for (int cur = 0;; cur ^= 1) {
        const bool more = BRUTE ? small_scene_iteration<COUNT, SPH64, ENV>(sc, rc, c, q, cur, accum, s_prims, s_u32, s_u64, env)
                                : wavefront_iteration<BRUTE, COUNT, SPH64, ENV>(sc, rc, c, q, cur, accum, s_stack, s_prims, s_u32, s_u64, env);
        if (!more) break;
    }
    if (threadIdx.x == 0) {
        atomicMax(&c->iterations, s_u64[4]);
        atomicAdd(&c->cyc_generate, s_u64[1]);
        atomicAdd(&c->cyc_extend, s_u64[2]);
        atomicAdd(&c->cyc_shade, s_u64[3]);
    }
}

template <bool BRUTE, bool COUNT, bool SPH64>
__global__ void __launch_bounds__(kBlock, SPH64 ? RRS_BLOCKS_PER_SM_F64 : RRS_BLOCKS_PER_SM) k_wavefront(DScene sc, RenderConst rc, DCounters* __restrict__ c,
                                                                      QueueSet q, float4* __restrict__ accum) {
    wavefront_kernel<BRUTE, COUNT, SPH64, false>(sc, rc, c, q, accum, nullptr);
}

// RRS_FLAG_ENV_SAMPLING: the same kernel with next-event estimation of the environment (separate instantiations, so
// that the code of the default form does not change)
template <bool BRUTE, bool COUNT, bool SPH64>
__global__ void __launch_bounds__(kBlock, SPH64 ? RRS_BLOCKS_PER_SM_F64 : RRS_BLOCKS_PER_SM) k_wavefront_env(DScene sc, RenderConst rc, DCounters* __restrict__ c,
                                                                          QueueSet q, float4* __restrict__ accum, DEnv env) {
    wavefront_kernel<BRUTE, COUNT, SPH64, true>(sc, rc, c, q, accum, &env);
}

// ---------------------------------------------------------------------------------------
// Register-resident path loop for small scenes (brute_count > 0: every sphere-series configuration).
// When the whole scene sits in 512 bytes of shared memory and a closest-hit query is a fixed 8-primitive
// loop, the HBM queues buy nothing: there is no long, divergent traversal to separate from shading, yet
// every ray still paid a 48-byte write, an 88-byte read-back, a hit record and two compaction passes
// (170 B/ray of DRAM traffic and ~45 % of DRAM bandwidth on the sphere series,
// profiles/r01b_c2_fused_metrics.csv).  Here a lane keeps ITS path in registers — generate, intersect,
// shade, next bounce — and takes a new path index the moment its path ends (path regeneration), so the
// warp stays full without any queue.  Same paths as the wavefront form (the RNG is keyed by pixel,
// sample and bounce), same accumulator, same census.  Warps claim path indices in chunks of 1024 from the
// global cursor (one global atomic per chunk) and hand them to their dead lanes by ballot/popc.
// ---------------------------------------------------------------------------------------
// Lanes of a warp are at different stages of their paths, and the four stages cost very differently
// (generate ~110 instructions, closest hit ~400, shade a hit ~450, shade a miss ~150).  Running all four
// every iteration with whatever lanes need them executed 22 of 32 lanes per instruction
// (profiles/r01g_c2_bench_metrics.csv).  Instead every lane carries its stage, and each iteration the warp
// runs ONE stage — the one most lanes are waiting for (four ballots + popc); the other lanes keep their
// state in registers and wait.  A stage's lane count only grows while it waits, so nothing starves.
enum PathStage : uint32_t { ST_GEN = 0, ST_ISECT = 1, ST_HIT = 2, ST_MISS = 3, ST_DONE = 4 };

template <bool COUNT, bool SPH64>
__global__ void __launch_bounds__(kBlock, SPH64 ? RRS_BLOCKS_PER_SM_F64 : RRS_BLOCKS_PER_SM)
k_pathloop(DScene sc, RenderConst rc, DCounters* __restrict__ c, float4* __restrict__ accum) {
    const uint32_t FULL = 0xFFFFFFFFu;
    __shared__ DPrim s_prims[RRS_BRUTE_MAX];
    stage_brute_prims(sc, s_prims);
    __syncthreads();
    const uint32_t lane = lane_id();
    const uint32_t lt_mask = (1u << lane) - 1u;
    const unsigned long long total = c->total_paths;
    unsigned long long w_next = 0, w_end = 0;  // this warp's claimed path range (warp-uniform)
    bool exhausted = false;                    // the global cursor has run past the end (warp-uniform)
    uint32_t stage = ST_GEN;
    float4 o4 = make_float4(0.f, 0.f, 0.f, 0.f), d4 = o4, st = o4;
    float2 h = make_float2(0.f, 0.f);
    double o64[3] = {0., 0., 0.};
    TravCounters cnt{0, 0};
    unsigned long long rays = 0, iters = 0;
    for (;;) {
        const uint32_t b_gen = __ballot_sync(FULL, stage == ST_GEN), b_is = __ballot_sync(FULL, stage == ST_ISECT);
        const uint32_t b_hit = __ballot_sync(FULL, stage == ST_HIT), b_miss = __ballot_sync(FULL, stage == ST_MISS);
        if ((b_gen | b_is | b_hit | b_miss) == 0u) break;
        const int n_gen = __popc(b_gen), n_is = __popc(b_is), n_hit = __popc(b_hit), n_miss = __popc(b_miss);
        ++iters;
        if (n_is >= n_gen && n_is >= n_hit && n_is >= n_miss) {
            // ---- extend: closest hit over the staged primitives ----
            if (stage == ST_ISECT) {
                uint32_t prim;
                closest_hit_brute<COUNT, SPH64>(sc, s_prims, xyz(o4), xyz(d4), __float_as_uint(o4.w), SPH64 ? o64 : nullptr, h.x, prim, cnt);
                h.y = __uint_as_float(prim);
                ++rays;
                stage = prim == RRS_NO_PRIM ? ST_MISS : ST_HIT;
            }
        } else if (n_hit >= n_gen && n_hit >= n_miss) {
            // ---- shade a hit: Material::evaluate, emission, Russian roulette ----
            if (stage == ST_HIT) {
                NextRay nr = shade_hit<SPH64, false>(sc, rc, accum, h, o4, d4, st, SPH64 ? o64 : nullptr);
                if (nr.alive) {
                    o4 = nr.no;
                    d4 = nr.nd;
                    st = nr.ns;
                    if (SPH64 && nr.carry64) {
                        o64[0] = nr.p64[0]; o64[1] = nr.p64[1]; o64[2] = nr.p64[2];
                    }
                    stage = ST_ISECT;
                } else {
                    stage = ST_GEN;
                }
            }
        } else if (n_miss >= n_gen) {
            // ---- shade a miss: background ----
            if (stage == ST_MISS) {
                shade_miss(sc, accum, d4, st);
                stage = ST_GEN;
            }
        } else {
            // ---- generate: waiting lanes take the next path indices of the warp's range ----
            if (w_next >= w_end && !exhausted) {
                unsigned long long base = 0;
                if (lane == 0) base = atomicAdd(&c->next_path, 1024ull);
                base = __shfl_sync(FULL, base, 0);
                w_next = base;
                w_end = base + 1024ull < total ? base + 1024ull : total;
                if (base >= total) {
                    exhausted = true;
                    w_end = w_next = 0;
                }
            }
            if (exhausted) {
                if (stage == ST_GEN) stage = ST_DONE;
            } else {
                const unsigned long long p = w_next + (unsigned long long)__popc(b_gen & lt_mask);
                if (stage == ST_GEN && p < w_end) {
                    uint32_t pixel = 0, sample = 0;
                    float3 d;
                    if (primary_ray(rc, p, pixel, sample, d)) {
                        o4 = make_float4(rc.cam.origin.x, rc.cam.origin.y, rc.cam.origin.z, __uint_as_float(RRS_NO_PRIM));
                        d4 = make_float4(d.x, d.y, d.z, __uint_as_float(pixel));
                        st = make_float4(1.f, 1.f, 1.f, __uint_as_float(sample << 8));
                        stage = ST_ISECT;
                    }
                }
                w_next += (unsigned long long)n_gen;
                if (w_next > w_end) w_next = w_end;
            }
        }
    }
    for (int o = 16; o > 0; o >>= 1) rays += __shfl_xor_sync(FULL, rays, o);
    if (lane == 0) {
        atomicAdd(&c->rays, rays);
        atomicMax(&c->iterations, iters);
    }
    flush_trav_counters<COUNT>(c, cnt);
}

// ---------------------------------------------------------------------------------------
// resolve: sum -> mean, NaN / negative census (rayrs/src/main.rs:81-89)
// ---------------------------------------------------------------------------------------
__global__ void k_resolve(const float4* __restrict__ accum, float* __restrict__ out, uint32_t npix, float inv_spp,
                          float expect_paths, unsigned long long* __restrict__ census) {
    uint32_t nan_cnt = 0, neg_cnt = 0, miss_cnt = 0;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < npix; i += gridDim.x * blockDim.x) {
        float4 a = __ldcs(accum + i);
        if (isnan(a.x) || isnan(a.y) || isnan(a.z)) nan_cnt++;
        if (a.x < 0.f || a.y < 0.f || a.z < 0.f) neg_cnt++;
        if (a.w != expect_paths) miss_cnt++;  // path census: every pixel must have terminated exactly spp_total paths
        out[3 * (size_t)i + 0] = a.x * inv_spp;
        out[3 * (size_t)i + 1] = a.y * inv_spp;
        out[3 * (size_t)i + 2] = a.z * inv_spp;
    }
    for (int o = 16; o > 0; o >>= 1) {
        nan_cnt += __shfl_xor_sync(0xFFFFFFFFu, nan_cnt, o);
        neg_cnt += __shfl_xor_sync(0xFFFFFFFFu, neg_cnt, o);
        miss_cnt += __shfl_xor_sync(0xFFFFFFFFu, miss_cnt, o);
    }
    if ((threadIdx.x & 31) == 0 && (nan_cnt | neg_cnt | miss_cnt)) {
        atomicAdd(census + 0, (unsigned long long)nan_cnt);
        atomicAdd(census + 1, (unsigned long long)neg_cnt);
        atomicAdd(census + 2, (unsigned long long)miss_cnt);
    }
}

// ---------------------------------------------------------------------------------------
// output stage: Image::to_raw_bytes (image.rs:193-222) fused with the division by spp.  f64 like the
// reference — it runs once per image, and the byte a pixel quantises to must not depend on fp32 pow.
// ---------------------------------------------------------------------------------------
__global__ void k_to_raw_bytes(const float4* __restrict__ accum, uint8_t* __restrict__ out, uint32_t npix, double inv_spp,
                               double gamma, unsigned long long* __restrict__ census) {
    uint32_t bright = 0, nan_cnt = 0, neg_cnt = 0;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < npix; i += gridDim.x * blockDim.x) {
        const float4 a = accum[i];
        // the f32 mean is the pixel value the host would hold (rrs_resolve); widen it like `val` in the reference
        const double v[3] = {(double)(a.x * (float)inv_spp), (double)(a.y * (float)inv_spp), (double)(a.z * (float)inv_spp)};
        if (isnan(v[0]) || isnan(v[1]) || isnan(v[2])) nan_cnt++;
        if (v[0] < 0. || v[1] < 0. || v[2] < 0.) neg_cnt++;
        if (v[0] > 1. || v[1] > 1. || v[2] > 1.) bright++;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            // Vector::clip vecmath.rs:389-397: x.min(1).max(0); f64::min drops a NaN operand, so NaN clips to 1.
            // Spelled out: nvcc folds fmax(fmin(x, 1), 0) into a form that lets the NaN through.
            double c = isnan(v[k]) ? 1. : (v[k] < 0. ? 0. : (v[k] > 1. ? 1. : v[k]));
            double q = 255.99 * pow(c, gamma);
            out[3 * (size_t)i + k] = (uint8_t)(q < 0. ? 0. : (q > 255. ? 255. : q));  // Rust `as u8` saturates
        }
    }
    for (int o = 16; o > 0; o >>= 1) {
        bright += __shfl_xor_sync(0xFFFFFFFFu, bright, o);
        nan_cnt += __shfl_xor_sync(0xFFFFFFFFu, nan_cnt, o);
        neg_cnt += __shfl_xor_sync(0xFFFFFFFFu, neg_cnt, o);
    }
    if ((threadIdx.x & 31) == 0 && (bright | nan_cnt | neg_cnt)) {
        atomicAdd(census + 0, (unsigned long long)bright);
        atomicAdd(census + 1, (unsigned long long)nan_cnt);
        atomicAdd(census + 2, (unsigned long long)neg_cnt);
    }
}

// ---------------------------------------------------------------------------------------
// probes (parity entry points)
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kBlock) k_intersect32(DScene sc, const float4* __restrict__ ray_o,
                                                         const float4* __restrict__ ray_d, uint32_t n,
                                                         int32_t* __restrict__ obj_id, float* __restrict__ t_out) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    uint32_t* s_stack = reinterpret_cast<uint32_t*>(smem_raw);
    __shared__ DPrim s_prims[RRS_BRUTE_MAX];
    stage_brute_prims(sc, s_prims);
    __syncthreads();
    SStack stack;
    stack.init(s_stack + threadIdx.x, blockDim.x);
    TravCounters cnt{0, 0};
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        float4 o4 = ldq(ray_o + i), d4 = ldq(ray_d + i);
        float t;
        uint32_t prim;
        if (sc.brute_count)
            closest_hit_brute<false, false>(sc, s_prims, xyz(o4), xyz(d4), RRS_NO_PRIM, nullptr, t, prim, cnt);
        else
            closest_hit<false, false>(sc, xyz(o4), xyz(d4), RRS_NO_PRIM, nullptr, stack, t, prim, cnt);
        t = refine_hit_t(sc, prim, xyz(o4), xyz(d4), t);
        if (prim == RRS_NO_PRIM) {
            obj_id[i] = -1;
            t_out[i] = INFINITY;
        } else {
            obj_id[i] = (int32_t)__float_as_uint(__ldg(reinterpret_cast<const float4*>(sc.prims + prim) + 1).w);
            t_out[i] = t;
        }
    }
}

template <bool STAGED>
__global__ void k_material_probe(DMat m, const float* __restrict__ nv, const float* __restrict__ u, uint32_t n,
                                 float* __restrict__ out) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float3 nrm = f3(nv[6 * i], nv[6 * i + 1], nv[6 * i + 2]);
    float3 view = f3(nv[6 * i + 3], nv[6 * i + 4], nv[6 * i + 5]);
    ScatterOut so = material_evaluate<STAGED>(m, nrm, view, u[3 * i], u[3 * i + 1], u[3 * i + 2]);
    float* o = out + 7 * (size_t)i;
    o[0] = so.scatter ? 1.f : 0.f;
    o[1] = so.color.x; o[2] = so.color.y; o[3] = so.color.z;
    o[4] = so.dir.x; o[5] = so.dir.y; o[6] = so.dir.z;
}

__global__ void k_background_probe(DScene sc, const float* __restrict__ dirs, uint32_t n, float* __restrict__ out) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float3 c = background(sc, f3(dirs[3 * i], dirs[3 * i + 1], dirs[3 * i + 2]));
    out[3 * i] = c.x; out[3 * i + 1] = c.y; out[3 * i + 2] = c.z;
}

__global__ void k_env_sample_probe(DScene sc, DEnv env, const float4* __restrict__ u, uint32_t n, float4* __restrict__ out) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float4 v = u[i];
    float3 d;
    const float pdf = env_sample(sc, env, v.x, v.y, v.z, v.w, d);
    out[i] = make_float4(d.x, d.y, d.z, pdf);
}

__global__ void k_env_pdf_probe(DScene sc, DEnv env, const float* __restrict__ dirs, uint32_t n, float* __restrict__ out) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    out[i] = env_pdf(sc, env, f3(dirs[3 * i], dirs[3 * i + 1], dirs[3 * i + 2]));
}

__global__ void k_rng_probe(uint64_t seed, uint32_t pixel, uint32_t sample, uint32_t slot, float* out) {
    float4 u = rng_uniforms(seed, pixel, sample, slot);
    out[0] = u.x; out[1] = u.y; out[2] = u.z; out[3] = u.w;
}

// ---------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------
static size_t extend_smem_bytes(const DScene& d) {
    return (size_t)d.stack_entries * kBlock * sizeof(uint32_t);  // per thread: one traversal stack
}

static void free_queues(Wavefront& w) {
    cudaFree(w.ray_o); cudaFree(w.ray_d); cudaFree(w.state); cudaFree(w.count); cudaFree(w.org64); cudaFree(w.hits); cudaFree(w.wmis);
    w.wmis = nullptr;
    w.ray_o = w.ray_d = w.state = nullptr;
    w.count = nullptr;
    w.org64 = nullptr;
    w.hits = nullptr;
    w.capacity = 0;
}

static int ensure_wavefront(SceneImpl* s, uint32_t regions, uint32_t region_cap, bool env, std::string& err) {
    Wavefront& w = s->wf;
    if (w.regions == regions && w.region_cap == region_cap && w.capacity && w.counters) {
        if (env && !w.wmis) RRS_CUDA_CHECK(cudaMalloc(&w.wmis, sizeof(float) * 2 * (size_t)w.capacity), err);
        return RRS_OK;
    }
    free_queues(w);
    const size_t cap = (size_t)regions * region_cap;
    RRS_CUDA_CHECK(cudaMalloc(&w.ray_o, sizeof(float4) * 2 * cap), err);
    RRS_CUDA_CHECK(cudaMalloc(&w.ray_d, sizeof(float4) * 2 * cap), err);
    RRS_CUDA_CHECK(cudaMalloc(&w.state, sizeof(float4) * 2 * cap), err);
    RRS_CUDA_CHECK(cudaMalloc(&w.count, sizeof(uint32_t) * 2 * regions), err);
    if (s->sphere64) RRS_CUDA_CHECK(cudaMalloc(&w.org64, sizeof(double) * 3 * 2 * cap), err);
    RRS_CUDA_CHECK(cudaMalloc(&w.hits, sizeof(float2) * cap), err);
    if (env) RRS_CUDA_CHECK(cudaMalloc(&w.wmis, sizeof(float) * 2 * cap), err);
    if (!w.counters) RRS_CUDA_CHECK(cudaMalloc(&w.counters, sizeof(DCounters)), err);
    if (!w.h_counters) RRS_CUDA_CHECK(cudaMallocHost(&w.h_counters, sizeof(DCounters)), err);
    w.capacity = (uint32_t)cap;
    w.regions = regions;
    w.region_cap = region_cap;
    return RRS_OK;
}

void wf_free(SceneImpl* s) {
    wf_finish_stats(s);  // an asynchronous render may still be running
    Wavefront& w = s->wf;
    free_queues(w);
    cudaFree(w.counters);
    if (w.h_counters) cudaFreeHost(w.h_counters);
    for (auto e : s->ev_pool) cudaEventDestroy(e);
    s->ev_pool.clear();
    w = Wavefront{};
}

static DCamera make_camera(const RrsCamera* c, uint32_t W, uint32_t H) {
    DCamera d;
    d.origin = make_float3((float)c->origin[0], (float)c->origin[1], (float)c->origin[2]);
    d.e_x = make_float3((float)c->e_x[0], (float)c->e_x[1], (float)c->e_x[2]);
    d.e_y = make_float3((float)c->e_y[0], (float)c->e_y[1], (float)c->e_y[2]);
    d.z = make_float3((float)c->z_scaled[0], (float)c->z_scaled[1], (float)c->z_scaled[2]);
    d.inv_ppc = (float)(1.0 / (double)c->ppc);
    d.half_w = (float)(c->width / 2.);
    d.half_h = (float)(c->height / 2.);
    d.W = W;
    d.H = H;
    return d;
}

int wf_render_accumulate(SceneImpl* s, const RrsCamera* cam, const RrsRenderParams* p, float4* d_accum,
                         cudaStream_t stream, std::string& err) {
    if (!cam || !p || !d_accum) { err = "null argument"; return RRS_ERR_INVALID; }
    if (p->width == 0 || p->height == 0) { err = "empty image"; return RRS_ERR_INVALID; }
    if (p->width != cam->x_pixels || p->height != cam->y_pixels) {
        err = "render size does not match Camera::x_pixels/y_pixels";
        return RRS_ERR_INVALID;
    }
    if (p->max_bounces > 255) { err = "max_bounces > 255 not supported"; return RRS_ERR_INVALID; }
    if ((unsigned long long)p->sample_offset + p->spp > (1ull << 24)) { err = "sample index exceeds 2^24"; return RRS_ERR_INVALID; }
    if ((unsigned long long)p->width * p->height > 0xFFFFFFFFull) { err = "image too large"; return RRS_ERR_INVALID; }
    const bool env = (p->flags & RRS_FLAG_ENV_SAMPLING) != 0;
    if (env && (p->flags & RRS_FLAG_SPLIT_KERNELS)) { err = "RRS_FLAG_ENV_SAMPLING runs in the fused kernel only (not with RRS_FLAG_SPLIT_KERNELS)"; return RRS_ERR_INVALID; }
    if (env && !s->env_ok) { err = "the environment map cannot be tabulated for sampling (non-finite texels)"; return RRS_ERR_INVALID; }
    RRS_CUDA_CHECK(cudaSetDevice(s->device), err);
    wf_finish_stats(s);  // a scene's queues and counters serve one render at a time
    // ---- launch geometry: every kernel runs `regions` blocks, block b owns queue stripe b ----
    const bool count = (p->flags & RRS_FLAG_COUNT_TRAVERSAL) != 0;
    const bool phases = (p->flags & RRS_FLAG_TIME_PHASES) != 0;
    const bool exact_tiles = (p->width % 8u == 0) && (p->height % 4u == 0);
    size_t smem = extend_smem_bytes(s->d);
    const bool sph64 = s->sphere64 != nullptr;
    const bool brute = s->d.brute_count > 0;
    const int sel = (brute ? 4 : 0) | (count ? 2 : 0) | (sph64 ? 1 : 0);
    typedef void (*ExtendFn)(DScene, DCounters*, QueueSet, int);
    static const ExtendFn etable[8] = {k_extend<false, false, false>, k_extend<false, false, true>,
                                       k_extend<false, true, false>,  k_extend<false, true, true>,
                                       k_extend<true, false, false>,  k_extend<true, false, true>,
                                       k_extend<true, true, false>,   k_extend<true, true, true>};
    ExtendFn extend_fn = etable[sel];
    auto shade_fn = sph64 ? k_shade<true> : k_shade<false>;
    typedef void (*PathFn)(DScene, RenderConst, DCounters*, float4*);
    static const PathFn ptable[4] = {k_pathloop<false, false>, k_pathloop<false, true>, k_pathloop<true, false>,
                                     k_pathloop<true, true>};
    PathFn path_fn = ptable[sel & 3];
    // the small-scene (brute force) and BVH forms of the fused kernel are separate instantiations: half the code
    // each (the SPH64 form with both was ~110 KB of SASS and stalled on instruction fetch, profiles/r01h_c3_*)
    typedef void (*FusedFn)(DScene, RenderConst, DCounters*, QueueSet, float4*);
    static const FusedFn table[8] = {k_wavefront<false, false, false>, k_wavefront<false, false, true>,
                                     k_wavefront<false, true, false>,  k_wavefront<false, true, true>,
                                     k_wavefront<true, false, false>,  k_wavefront<true, false, true>,
                                     k_wavefront<true, true, false>,   k_wavefront<true, true, true>};
    FusedFn fused_fn = table[sel];
    typedef void (*EnvFusedFn)(DScene, RenderConst, DCounters*, QueueSet, float4*, DEnv);
    static const EnvFusedFn env_table[8] = {k_wavefront_env<false, false, false>, k_wavefront_env<false, false, true>,
                                            k_wavefront_env<false, true, false>,  k_wavefront_env<false, true, true>,
                                            k_wavefront_env<true, false, false>,  k_wavefront_env<true, false, true>,
                                            k_wavefront_env<true, true, false>,   k_wavefront_env<true, true, true>};
    EnvFusedFn env_fn = env_table[sel];
    const void* fused_kernel = env ? (const void*)env_fn : (const void*)fused_fn;
    RRS_CUDA_CHECK(cudaFuncSetAttribute(fused_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem), err);
    auto generate_fn = k_generate;
    RRS_CUDA_CHECK(cudaFuncSetAttribute(extend_fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem), err);
    int occ_ext = 0, occ_shade = 0;
    RRS_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_ext, extend_fn, kBlock, smem), err);
    RRS_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_shade, shade_fn, kBlock, 0), err);
    int occ_fused = 0;
    RRS_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_fused, fused_kernel, kBlock, smem), err);
    if (occ_ext < 1 || occ_shade < 1 || occ_fused < 1) { err = "kernel does not fit on an SM (traversal stack too deep)"; return RRS_ERR_TOO_DEEP; }
    if (!(p->flags & RRS_FLAG_SPLIT_KERNELS)) occ_ext = occ_shade = occ_fused;
    // one wave of the most register-hungry kernel: all stripes are resident at once
    const uint32_t regions = (uint32_t)s->num_sms * (uint32_t)std::min(occ_ext, occ_shade);
    // rays in flight: 4M for the small-scene form, 8M for the BVH form (fewer, longer iterations: configuration 5 +2 %,
    // configuration 4 +1.5 % over 4M; 16M / 32M within 1 % of 8M — profiles/ab_logs/queue_r02x.log)
    uint32_t want = p->queue_capacity ? p->queue_capacity : (brute ? (1u << 22) : (1u << 23));
    uint32_t region_cap = std::max(32u, ((want + regions - 1) / regions + 31u) & ~31u);
    // environment sampling: as many paths in flight, and room for a shadow ray beside each continuation
    if (env) region_cap *= 2u;
    int rc_ = ensure_wavefront(s, regions, region_cap, env, err);
    if (rc_ != RRS_OK) return rc_;
    Wavefront& w = s->wf;
    RRS_CUDA_CHECK(cudaMemsetAsync(w.count, 0, sizeof(uint32_t) * 2 * regions, stream), err);
    QueueSet q;
    q.ray_o = w.ray_o;
    q.ray_d = w.ray_d;
    q.state = w.state;
    q.hits = w.hits;
    q.count = w.count;
    q.org64 = w.org64;
    q.capacity = w.capacity;
    q.regions = regions;
    q.region_cap = region_cap;

    RenderConst rc;
    rc.cam = make_camera(cam, p->width, p->height);
    rc.cam64 = *cam;
    rc.tiles_x = (p->width + 7u) / 8u;
    rc.tiles_y = (p->height + 3u) / 4u;
    rc.exact_tiles = exact_tiles ? 1u : 0u;
    rc.npix_pad = (unsigned long long)rc.tiles_x * rc.tiles_y * 32ull;
    // floor(2^32 / d): __umulhi(n, magic) is floor(n / d) or one less for every n < 2^32 (corrected on the device)
    rc.small_index = (rc.npix_pad * (unsigned long long)p->spp < (1ull << 32)) ? 1u : 0u;
    rc.tiles = rc.tiles_x * rc.tiles_y;
    rc.magic_tiles = (uint32_t)std::min<unsigned long long>((1ull << 32) / rc.tiles, 0xFFFFFFFFull);
    // samples of one tile generated back to back: the largest power of two <= 2^RRS_SAMPLE_BLOCK_LOG2 that divides spp
    rc.sblk_shift = 0;
    while (rc.sblk_shift < RRS_SAMPLE_BLOCK_LOG2 && (p->spp >> rc.sblk_shift) % 2u == 0u && (p->spp >> rc.sblk_shift) > 1u) ++rc.sblk_shift;
    rc.magic_tiles_y = (uint32_t)std::min<unsigned long long>((1ull << 32) / rc.tiles_y, 0xFFFFFFFFull);
    // stripe width in tiles: the largest power of two <= 2^RRS_TILE_STRIPE_LOG2 that divides tiles_x
    rc.ws_shift = 0;
    while (rc.ws_shift < RRS_TILE_STRIPE_LOG2 && (rc.tiles_x >> rc.ws_shift) % 2u == 0u && (rc.tiles_x >> rc.ws_shift) > 1u) ++rc.ws_shift;
    rc.spp = p->spp;
    rc.sample_offset = p->sample_offset;
    rc.max_bounces = p->max_bounces;
    rc.seed = p->seed;

    DCounters init{};
    init.total_paths = rc.npix_pad * (unsigned long long)p->spp;
    if (p->max_bounces == 0) init.total_paths = 0;  // radiance() with 0 bounces returns black
    // pageable source: the runtime stages it before the call returns, so `init` may die with this frame
    RRS_CUDA_CHECK(cudaMemcpyAsync(w.counters, &init, sizeof(DCounters), cudaMemcpyHostToDevice, stream), err);

    // ---- L2 residency ------------------------------------------------------------------------
    // The traversal's node / primitive fetches are the only traffic with reuse; the ray, state and hit queues stream
    // (written once, read once, ld/st.global.cs) and the accumulator is touched once per path.  Without help the
    // queue streams evict the tree: the 1M-triangle scene (20 MB of nodes + 64 MB of primitives, smaller than the
    // 126 MB L2) ran at a 56 % L2 hit rate and 181 B of DRAM reads per ray (profiles/r01o_c4_wavefront_metrics.csv).
    // An access-policy window marks the top of the tree persisting: the first kL2PinBytes of the node array (numbered
    // breadth-first at the top, depth-first below), with a set-aside of exactly that size.
    // The set-aside (cudaLimitPersistingL2CacheSize) is a device-wide limit and every byte of it is lost to all other
    // traffic, so it is sized to what is pinned, claimed by a render that pins a tree and released by one that does
    // not (small scenes: their queues want the whole L2); it is touched only when its size on the device changes.
    // Measured (profiles/ab_logs/ab_r02x_l2_set_aside_size.log, l2window_r02x_window_vs_none.log): round 2's first
    // form — the device maximum set aside, [nodes | primitives] or all nodes pinned — was 1.3 % (config 4) and 7.7 %
    // (config 5) SLOWER than no window at all; 8 / 24 / 48 MB set aside and pinned are +0.2 % / +0.6 % over none.
    constexpr size_t kL2PinBytes = 32u << 20;
    bool window_set = false;
    const bool want_window = !brute && s->l2_persist_bytes && s->geom_blob && !(p->flags & RRS_FLAG_NO_L2_WINDOW);
    const size_t pin_bytes = std::min(std::min(s->node_bytes, kL2PinBytes), std::min(s->l2_persist_bytes, s->l2_window_max));
    bool set_aside_ok = false;
    if (s->l2_persist_bytes && s->device >= 0 && s->device < kMaxDevices) {
        const size_t want = want_window ? pin_bytes : 0;
        std::atomic<size_t>& cur = g_l2_set_aside[s->device];
        if (cur.load() != want) {
            const bool ok = cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, want) == cudaSuccess;
            cudaGetLastError();
            cur.store(ok ? want : kUnknownSetAside);
        }
        set_aside_ok = cur.load() == want;
    }
    if (want_window && set_aside_ok && pin_bytes) {
        cudaStreamAttrValue av{};
        av.accessPolicyWindow.base_ptr = s->geom_blob;
        av.accessPolicyWindow.num_bytes = pin_bytes;
        av.accessPolicyWindow.hitRatio = 1.f;
        av.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
        av.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
        window_set = cudaStreamSetAttribute(stream, cudaStreamAttributeAccessPolicyWindow, &av) == cudaSuccess;
        cudaGetLastError();
    }
    auto clear_window = [&]() {
        if (!window_set) return;
        cudaStreamAttrValue av{};
        av.accessPolicyWindow.num_bytes = 0;  // launches after this one run without a window
        cudaStreamSetAttribute(stream, cudaStreamAttributeAccessPolicyWindow, &av);
        cudaGetLastError();
    };

    // event pool: [0]=start [1]=stop, then 5 per iteration when phase timing is on
    auto get_event = [&](size_t idx) -> cudaEvent_t {
        while (s->ev_pool.size() <= idx) {
            cudaEvent_t e;
            cudaEventCreate(&e);
            s->ev_pool.push_back(e);
        }
        return s->ev_pool[idx];
    };
    cudaEvent_t ev_start = get_event(0), ev_stop = get_event(1);
    RRS_CUDA_CHECK(cudaEventRecord(ev_start, stream), err);

    uint64_t launches = 0;
    s->phase_ev.clear();
    const bool split = (p->flags & RRS_FLAG_SPLIT_KERNELS) != 0;
    // The register-resident path loop beat the queued kernel by 16 % while that still ran a separate extend phase
    // (profiles/ab_logs/sweep_pathloop.log); with the closest hit fused into the shade phase the queued kernel is as
    // fast or faster on every small scene (plastic series +5 %, sweep_pl_vs_q.log) — compaction gives it full warps
    // every iteration — so the path loop is an option (RRS_FLAG_FORCE_PATHLOOP), not the default.
    const bool want_pathloop = (p->flags & RRS_FLAG_FORCE_PATHLOOP) != 0;
    const bool pathloop = !split && brute && want_pathloop && !(p->flags & RRS_FLAG_FORCE_QUEUES) && !env;
    if (pathloop) {
        // small scene: register-resident paths, no queues (k_pathloop)
        int occ_path = 0;
        RRS_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_path, path_fn, kBlock, 0), err);
        path_fn<<<(uint32_t)s->num_sms * (uint32_t)std::max(occ_path, 1), kBlock, 0, stream>>>(s->d, rc, w.counters, d_accum);
        launches = 1;
        RRS_CUDA_CHECK(cudaGetLastError(), err);
    } else if (env) {
        DEnv e = s->env;
        e.wmis = w.wmis;
        env_fn<<<regions, kBlock, smem, stream>>>(s->d, rc, w.counters, q, d_accum, e);
        launches = 1;
        RRS_CUDA_CHECK(cudaGetLastError(), err);
    } else if (!split) {
        // one persistent launch for the whole render
        fused_fn<<<regions, kBlock, smem, stream>>>(s->d, rc, w.counters, q, d_accum);
        launches = 1;
        RRS_CUDA_CHECK(cudaGetLastError(), err);
    } else {
        // per-phase profiling form: the host polls the `done` flag, so this branch blocks
        int cur = 0;
        const uint32_t chunk = 8;
        size_t ev_next = 2;
        bool done = false;
        while (!done) {
            for (uint32_t k = 0; k < chunk; ++k) {
                int nxt = cur ^ 1;
                size_t e0 = 0;
                if (phases) {
                    e0 = ev_next;
                    ev_next += 5;
                    get_event(e0 + 4);
                    s->phase_ev.push_back(e0);
                    cudaEventRecord(s->ev_pool[e0], stream);
                }
                k_plan<<<1, 32, 0, stream>>>(w.counters);
                if (phases) cudaEventRecord(s->ev_pool[e0 + 1], stream);
                generate_fn<<<regions, kBlock, 0, stream>>>(rc, w.counters, q, cur);
                if (phases) cudaEventRecord(s->ev_pool[e0 + 2], stream);
                extend_fn<<<regions, kBlock, smem, stream>>>(s->d, w.counters, q, cur);
                if (phases) cudaEventRecord(s->ev_pool[e0 + 3], stream);
                shade_fn<<<regions, kBlock, 0, stream>>>(s->d, rc, w.counters, q, cur, d_accum);
                if (phases) cudaEventRecord(s->ev_pool[e0 + 4], stream);
                launches += 4;
                cur = nxt;
            }
            RRS_CUDA_CHECK(cudaMemcpyAsync(w.h_counters, w.counters, sizeof(DCounters), cudaMemcpyDeviceToHost, stream), err);
            RRS_CUDA_CHECK(cudaStreamSynchronize(stream), err);
            RRS_CUDA_CHECK(cudaGetLastError(), err);
            done = w.h_counters->done != 0;
        }
    }
    clear_window();
    RRS_CUDA_CHECK(cudaMemcpyAsync(w.h_counters, w.counters, sizeof(DCounters), cudaMemcpyDeviceToHost, stream), err);
    RRS_CUDA_CHECK(cudaEventRecord(ev_stop, stream), err);
    // not synchronised: the statistics are completed by wf_finish_stats (rrs_stats, rrs_resolve, the next render)
    s->stats = RrsStats{};
    s->stats.kernel_launches = launches;
    s->stats.paths = (uint64_t)p->width * p->height * p->spp;
    s->stats.kernel_form = pathloop ? RRS_FORM_PATHLOOP : (split ? RRS_FORM_SPLIT : RRS_FORM_WAVEFRONT);
    s->stats_pending = true;
    s->pending_split = split;
    s->pending_phases = phases;
    s->pending_window = window_set;
    return RRS_OK;
}

void wf_finish_stats(SceneImpl* s) {
    if (!s->stats_pending) return;
    s->stats_pending = false;
    cudaSetDevice(s->device);
    if (s->ev_pool.size() < 2 || cudaEventSynchronize(s->ev_pool[1]) != cudaSuccess) {
        cudaGetLastError();
        return;
    }
    if (s->pending_window) {
        cudaCtxResetPersistingL2Cache();  // hand the carve-out back: the next launch may be a different scene's
        cudaGetLastError();
    }
    Wavefront& w = s->wf;
    float ms = 0.f;
    cudaEventElapsedTime(&ms, s->ev_pool[0], s->ev_pool[1]);
    RrsStats& st = s->stats;
    st.rays = w.h_counters->rays;
    st.iterations = w.h_counters->iterations;
    st.device_ms = ms;
    st.nodes_visited = w.h_counters->nodes_visited;
    st.prims_tested = w.h_counters->prims_tested;
    st.generate_ms = st.extend_ms = st.shade_ms = 0.;
    if (!s->pending_split) {
        // per-phase share of the fused kernel from its in-kernel cycle counters (summed over blocks)
        double cg = (double)w.h_counters->cyc_generate, ce = (double)w.h_counters->cyc_extend, cs = (double)w.h_counters->cyc_shade;
        double tot = cg + ce + cs;
        if (tot > 0) {
            st.generate_ms = ms * cg / tot;
            st.extend_ms = ms * ce / tot;
            st.shade_ms = ms * cs / tot;
        }
    } else if (s->pending_phases) {
        double g = 0, e = 0, sh = 0;
        for (size_t e0 : s->phase_ev) {
            float a = 0, b = 0, c2 = 0;
            cudaEventElapsedTime(&a, s->ev_pool[e0 + 1], s->ev_pool[e0 + 2]);
            cudaEventElapsedTime(&b, s->ev_pool[e0 + 2], s->ev_pool[e0 + 3]);
            cudaEventElapsedTime(&c2, s->ev_pool[e0 + 3], s->ev_pool[e0 + 4]);
            g += a; e += b; sh += c2;
        }
        st.generate_ms = g;
        st.extend_ms = e;
        st.shade_ms = sh;
    }
}

int wf_resolve(SceneImpl* s, const float4* d_accum, uint32_t w, uint32_t h, uint32_t spp_total, float* out,
               bool out_is_device, cudaStream_t stream, std::string& err) {
    if (!d_accum || !out || spp_total == 0) { err = "bad resolve argument"; return RRS_ERR_INVALID; }
    if (w == 0 || h == 0 || (unsigned long long)w * h > 0xFFFFFFFFull) { err = "bad image size"; return RRS_ERR_INVALID; }
    RRS_CUDA_CHECK(cudaSetDevice(s->device), err);
    const uint32_t npix = w * h;
    const size_t bytes = sizeof(float) * 3 * (size_t)npix;
    if (!s->census) {
        RRS_CUDA_CHECK(cudaMalloc(&s->census, 3 * sizeof(unsigned long long)), err);
        RRS_CUDA_CHECK(cudaMallocHost(&s->h_census, 3 * sizeof(unsigned long long)), err);
    }
    RRS_CUDA_CHECK(cudaMemsetAsync(s->census, 0, 3 * sizeof(unsigned long long), stream), err);
    float* d_out = out;
    bool direct = false;  // the caller's host buffer is page-locked: DMA straight into it
    if (!out_is_device) {
        cudaPointerAttributes at;
        if (cudaPointerGetAttributes(&at, out) == cudaSuccess) direct = at.type == cudaMemoryTypeHost;
        cudaGetLastError();  // an unregistered pointer is not an error here
        // persistent device image (+ pinned staging buffer for pageable destinations): the host copy is one async D2H
        if (s->resolve_bytes < bytes) {
            cudaFree(s->resolve_dev);
            if (s->resolve_pinned) cudaFreeHost(s->resolve_pinned);
            s->resolve_dev = nullptr;
            s->resolve_pinned = nullptr;
            s->resolve_bytes = 0;
            RRS_CUDA_CHECK(cudaMalloc(&s->resolve_dev, bytes), err);
            RRS_CUDA_CHECK(cudaMallocHost(&s->resolve_pinned, bytes), err);
            s->resolve_bytes = bytes;
        }
        d_out = s->resolve_dev;
    }
    int grid = std::min<uint32_t>((npix + 255) / 256, (uint32_t)s->num_sms * 8u);
    k_resolve<<<grid, 256, 0, stream>>>(d_accum, d_out, npix, 1.0f / (float)spp_total, (float)spp_total, s->census);
    if (!out_is_device)
        RRS_CUDA_CHECK(cudaMemcpyAsync(direct ? out : s->resolve_pinned, d_out, bytes, cudaMemcpyDeviceToHost, stream), err);
    RRS_CUDA_CHECK(cudaMemcpyAsync(s->h_census, s->census, 3 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, stream), err);
    RRS_CUDA_CHECK(cudaStreamSynchronize(stream), err);
    if (!out_is_device && !direct) std::memcpy(out, s->resolve_pinned, bytes);
    wf_finish_stats(s);
    s->stats.nan_pixels = s->h_census[0];
    s->stats.negative_pixels = s->h_census[1];
    s->stats.census_mismatch_pixels = s->h_census[2];
    s->stats.kernel_launches += 1;
    return RRS_OK;
}

int wf_to_raw_bytes(SceneImpl* s, const float4* d_accum, uint32_t w, uint32_t h, uint32_t spp_total, double gamma,
                    uint8_t* out, bool out_is_device, cudaStream_t stream, uint64_t* census3, std::string& err) {
    if (!d_accum || !out || spp_total == 0) { err = "bad to_raw_bytes argument"; return RRS_ERR_INVALID; }
    if (w == 0 || h == 0 || (unsigned long long)w * h > 0xFFFFFFFFull) { err = "bad image size"; return RRS_ERR_INVALID; }
    RRS_CUDA_CHECK(cudaSetDevice(s->device), err);
    const uint32_t npix = w * h;
    const size_t bytes = 3 * (size_t)npix;
    DevBuf<unsigned long long> d_census;
    DevBuf<uint8_t> d_stage;
    uint8_t* d_out = out;
    RRS_CUDA_CHECK(d_census.alloc(3), err);
    RRS_CUDA_CHECK(cudaMemsetAsync(d_census, 0, 3 * sizeof(unsigned long long), stream), err);
    if (!out_is_device) {
        RRS_CUDA_CHECK(d_stage.alloc(bytes), err);
        d_out = d_stage;
    }
    int grid = std::min<uint32_t>((npix + 255) / 256, (uint32_t)s->num_sms * 8u);
    k_to_raw_bytes<<<grid, 256, 0, stream>>>(d_accum, d_out, npix, 1.0 / (double)spp_total, gamma, d_census);
    RRS_CUDA_CHECK(cudaGetLastError(), err);
    unsigned long long hc[3] = {0, 0, 0};
    if (!out_is_device) RRS_CUDA_CHECK(cudaMemcpyAsync(out, d_out, bytes, cudaMemcpyDeviceToHost, stream), err);
    RRS_CUDA_CHECK(cudaMemcpyAsync(hc, d_census, sizeof(hc), cudaMemcpyDeviceToHost, stream), err);
    RRS_CUDA_CHECK(cudaStreamSynchronize(stream), err);
    if (census3) { census3[0] = hc[0]; census3[1] = hc[1]; census3[2] = hc[2]; }
    return RRS_OK;
}

int wf_intersect32(SceneImpl* s, const RrsRay* rays, size_t n, int32_t* obj_id, double* t, std::string& err) {
    RRS_CUDA_CHECK(cudaSetDevice(s->device), err);
    if (n == 0) return RRS_OK;
    if (n > 0x7FFFFFFFull) { err = "too many rays"; return RRS_ERR_INVALID; }
    std::vector<float4> ho(n), hd(n);
    for (size_t i = 0; i < n; ++i) {
        ho[i] = make_float4((float)rays[i].origin[0], (float)rays[i].origin[1], (float)rays[i].origin[2], 0.f);
        hd[i] = make_float4((float)rays[i].direction[0], (float)rays[i].direction[1], (float)rays[i].direction[2], 0.f);
    }
    DevBuf<float4> d_o, d_d;
    DevBuf<int32_t> d_id;
    DevBuf<float> d_t;
    RRS_CUDA_CHECK(d_o.alloc(n), err);
    RRS_CUDA_CHECK(d_d.alloc(n), err);
    RRS_CUDA_CHECK(d_id.alloc(n), err);
    RRS_CUDA_CHECK(d_t.alloc(n), err);
    RRS_CUDA_CHECK(cudaMemcpy(d_o, ho.data(), sizeof(float4) * n, cudaMemcpyHostToDevice), err);
    RRS_CUDA_CHECK(cudaMemcpy(d_d, hd.data(), sizeof(float4) * n, cudaMemcpyHostToDevice), err);
    size_t smem = extend_smem_bytes(s->d);
    RRS_CUDA_CHECK(cudaFuncSetAttribute(k_intersect32, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem), err);
    int grid = (int)std::min<size_t>((n + kBlock - 1) / kBlock, (size_t)s->num_sms * 8);
    k_intersect32<<<grid, kBlock, smem>>>(s->d, d_o, d_d, (uint32_t)n, d_id, d_t);
    RRS_CUDA_CHECK(cudaGetLastError(), err);
    std::vector<float> ht(n);
    RRS_CUDA_CHECK(cudaMemcpy(obj_id, d_id, sizeof(int32_t) * n, cudaMemcpyDeviceToHost), err);
    RRS_CUDA_CHECK(cudaMemcpy(ht.data(), d_t, sizeof(float) * n, cudaMemcpyDeviceToHost), err);
    for (size_t i = 0; i < n; ++i) t[i] = (double)ht[i];
    return RRS_OK;
}

int wf_material_evaluate(SceneImpl* s, uint32_t material, const double* nv, const double* u, size_t n, float* out,
                         std::string& err) {
    RRS_CUDA_CHECK(cudaSetDevice(s->device), err);
    const bool cases_form = (material & RRS_MATERIAL_FORM_CASES) != 0;
    material &= ~RRS_MATERIAL_FORM_CASES;
    if (material >= s->d.n_mats) { err = "material index out of range"; return RRS_ERR_INVALID; }
    if (n == 0) return RRS_OK;
    DMat m;
    RRS_CUDA_CHECK(cudaMemcpy(&m, s->mats + material, sizeof(DMat), cudaMemcpyDeviceToHost), err);
    std::vector<float> hnv(6 * n), hu(3 * n);
    for (size_t i = 0; i < 6 * n; ++i) hnv[i] = (float)nv[i];
    for (size_t i = 0; i < 3 * n; ++i) hu[i] = (float)u[i];
    DevBuf<float> d_nv, d_u, d_out;
    RRS_CUDA_CHECK(d_nv.alloc(6 * n), err);
    RRS_CUDA_CHECK(d_u.alloc(3 * n), err);
    RRS_CUDA_CHECK(d_out.alloc(7 * n), err);
    RRS_CUDA_CHECK(cudaMemcpy(d_nv, hnv.data(), sizeof(float) * 6 * n, cudaMemcpyHostToDevice), err);
    RRS_CUDA_CHECK(cudaMemcpy(d_u, hu.data(), sizeof(float) * 3 * n, cudaMemcpyHostToDevice), err);
    if (cases_form) k_material_probe<false><<<(unsigned)((n + 127) / 128), 128>>>(m, d_nv, d_u, (uint32_t)n, d_out);
    else k_material_probe<true><<<(unsigned)((n + 127) / 128), 128>>>(m, d_nv, d_u, (uint32_t)n, d_out);
    RRS_CUDA_CHECK(cudaGetLastError(), err);
    RRS_CUDA_CHECK(cudaMemcpy(out, d_out, sizeof(float) * 7 * n, cudaMemcpyDeviceToHost), err);
    return RRS_OK;
}

int wf_background(SceneImpl* s, const double* dirs, size_t n, float* out, std::string& err) {
    RRS_CUDA_CHECK(cudaSetDevice(s->device), err);
    if (n == 0) return RRS_OK;
    std::vector<float> hd(3 * n);
    for (size_t i = 0; i < 3 * n; ++i) hd[i] = (float)dirs[i];
    DevBuf<float> d_d, d_out;
    RRS_CUDA_CHECK(d_d.alloc(3 * n), err);
    RRS_CUDA_CHECK(d_out.alloc(3 * n), err);
    RRS_CUDA_CHECK(cudaMemcpy(d_d, hd.data(), sizeof(float) * 3 * n, cudaMemcpyHostToDevice), err);
    k_background_probe<<<(unsigned)((n + 127) / 128), 128>>>(s->d, d_d, (uint32_t)n, d_out);
    RRS_CUDA_CHECK(cudaGetLastError(), err);
    RRS_CUDA_CHECK(cudaMemcpy(out, d_out, sizeof(float) * 3 * n, cudaMemcpyDeviceToHost), err);
    return RRS_OK;
}

int wf_env_sample(SceneImpl* s, const double* u, size_t n, double* dir_pdf, std::string& err) {
    if (!s->env_ok) { err = "the environment map cannot be tabulated for sampling (non-finite texels)"; return RRS_ERR_INVALID; }
    if (!s->env.marg) { err = "the environment map is black: nothing to sample"; return RRS_ERR_INVALID; }
    RRS_CUDA_CHECK(cudaSetDevice(s->device), err);
    if (n == 0) return RRS_OK;
    if (n > 0x7FFFFFFFull) { err = "too many samples"; return RRS_ERR_INVALID; }
    // each uniform in [0, 1) as the device draws it: 24 bits that pick the cell + 24 more (hi, lo: env_sample)
    std::vector<float4> hu(n);
    auto split = [](double v, float& hi, float& lo) {
        const double x = std::ldexp(std::min(std::max(v, 0.), 1.), 24);
        const double f = std::min(std::floor(x), 16777215.);
        hi = (float)std::ldexp(f, -24);
        lo = (float)std::min(x - f, 1.);
    };
    for (size_t i = 0; i < n; ++i) {
        split(u[2 * i], hu[i].x, hu[i].z);
        split(u[2 * i + 1], hu[i].y, hu[i].w);
    }
    DevBuf<float4> d_u, d_out;
    RRS_CUDA_CHECK(d_u.alloc(n), err);
    RRS_CUDA_CHECK(d_out.alloc(n), err);
    RRS_CUDA_CHECK(cudaMemcpy(d_u, hu.data(), sizeof(float4) * n, cudaMemcpyHostToDevice), err);
    k_env_sample_probe<<<(unsigned)((n + 127) / 128), 128>>>(s->d, s->env, d_u, (uint32_t)n, d_out);
    RRS_CUDA_CHECK(cudaGetLastError(), err);
    std::vector<float4> ho(n);
    RRS_CUDA_CHECK(cudaMemcpy(ho.data(), d_out, sizeof(float4) * n, cudaMemcpyDeviceToHost), err);
    for (size_t i = 0; i < n; ++i) {
        dir_pdf[4 * i] = ho[i].x; dir_pdf[4 * i + 1] = ho[i].y; dir_pdf[4 * i + 2] = ho[i].z; dir_pdf[4 * i + 3] = ho[i].w;
    }
    return RRS_OK;
}

int wf_env_pdf(SceneImpl* s, const double* dirs, size_t n, double* pdf, std::string& err) {
    if (!s->env_ok) { err = "the environment map cannot be tabulated for sampling (non-finite texels)"; return RRS_ERR_INVALID; }
    RRS_CUDA_CHECK(cudaSetDevice(s->device), err);
    if (n == 0) return RRS_OK;
    if (n > 0x7FFFFFFFull) { err = "too many directions"; return RRS_ERR_INVALID; }
    std::vector<float> hd(3 * n);
    for (size_t i = 0; i < 3 * n; ++i) hd[i] = (float)dirs[i];
    DevBuf<float> d_d, d_out;
    RRS_CUDA_CHECK(d_d.alloc(3 * n), err);
    RRS_CUDA_CHECK(d_out.alloc(n), err);
    RRS_CUDA_CHECK(cudaMemcpy(d_d, hd.data(), sizeof(float) * 3 * n, cudaMemcpyHostToDevice), err);
    k_env_pdf_probe<<<(unsigned)((n + 127) / 128), 128>>>(s->d, s->env, d_d, (uint32_t)n, d_out);
    RRS_CUDA_CHECK(cudaGetLastError(), err);
    std::vector<float> ho(n);
    RRS_CUDA_CHECK(cudaMemcpy(ho.data(), d_out, sizeof(float) * n, cudaMemcpyDeviceToHost), err);
    for (size_t i = 0; i < n; ++i) pdf[i] = ho[i];
    return RRS_OK;
}

int wf_rng_uniforms(SceneImpl* s, uint64_t seed, uint32_t pixel, uint32_t sample, uint32_t slot, float* out4,
                    std::string& err) {
    RRS_CUDA_CHECK(cudaSetDevice(s->device), err);
    DevBuf<float> d;
    RRS_CUDA_CHECK(d.alloc(4), err);
    k_rng_probe<<<1, 1>>>(seed, pixel, sample, slot, d);
    RRS_CUDA_CHECK(cudaGetLastError(), err);
    RRS_CUDA_CHECK(cudaMemcpy(out4, d, 4 * sizeof(float), cudaMemcpyDeviceToHost), err);
    return RRS_OK;
}

}  // namespace rrs
