/* rayrs_b200.h — C ABI of the B200 path-tracing backend for rayrs.
 *
 * This is the drop-in boundary.  The reference (Frojdholm/rayrs) has no FFI of its own; the
 * seam this library replaces is the body of the rayon closure in rayrs/src/main.rs:61-94
 * (pixel x spp loop calling Camera::generate_primary_ray lib.rs:202-210 and radiance
 * lib.rs:521-560).  A Rust shim `rayrs_lib::gpu::render_gpu(&Camera, &Scene, spp,
 * max_bounces) -> Image` binds exactly these symbols (INTEGRATION.md shows the stub); the
 * C++ host mirror in rayrs_b200/host binds them the same way.
 *
 * Conventions
 *  - plain C types only; every pointer is borrowed for the duration of the call;
 *  - every entry point returns RRS_OK (0) or a negative RrsStatus and never unwinds;
 *    rrs_last_error() returns the message of the calling thread's last failure;
 *  - the reference panics on bad construction (assert!, e.g. geometry.rs:97,205-212;
 *    lib.rs:234-235): the same conditions return RRS_ERR_INVALID here and the shim turns
 *    a non-zero status into a panic;
 *  - there is NO CPU fallback: with no usable CUDA device every call that needs one
 *    fails with RRS_ERR_NO_DEVICE.
 */
#ifndef RAYRS_B200_H
#define RAYRS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RRS_ABI_VERSION 2

typedef enum RrsStatus {
    RRS_OK = 0,
    RRS_ERR_INVALID = -1,   /* bad argument / scene description (reference: assert! panic)   */
    RRS_ERR_NO_DEVICE = -2, /* no CUDA device, or not an sm_100 part                          */
    RRS_ERR_CUDA = -3,      /* CUDA runtime failure (message carries cudaGetErrorString)      */
    RRS_ERR_TOO_DEEP = -4,  /* BVH deeper than the traversal stack (RRS_MAX_STACK)            */
    RRS_ERR_NOMEM = -5,
    RRS_ERR_COMM = -6       /* NCCL missing (libnccl.so.2 could not be loaded) or an NCCL call failed */
} RrsStatus;

/* Primitive kinds: the three Hittable impls reachable from the scene API
 * (geometry.rs:72-157 Sphere, :159-304 Plane, :306-392 Triangle). */
typedef enum RrsPrimType { RRS_SPHERE = 0, RRS_PLANE = 1, RRS_TRIANGLE = 2 } RrsPrimType;

/* enum Axis, geometry.rs:159-167 (declaration order). */
typedef enum RrsAxis { RRS_AXIS_X = 0, RRS_AXIS_XREV = 1, RRS_AXIS_Y = 2, RRS_AXIS_YREV = 3, RRS_AXIS_Z = 4, RRS_AXIS_ZREV = 5 } RrsAxis;

/* enum Material, material.rs:57-68 (declaration order). */
typedef enum RrsMaterialTag {
    RRS_MAT_LAMBERTIAN = 0,
    RRS_MAT_REFLECT = 1,
    RRS_MAT_REFRACT = 2,
    RRS_MAT_GLASS = 3,
    RRS_MAT_COOK_TORRANCE = 4,
    RRS_MAT_COOK_TORRANCE_REFRACT = 5,
    RRS_MAT_COOK_TORRANCE_GLASS = 6,
    RRS_MAT_PLASTIC = 7,
    RRS_MAT_NO_REFLECT = 8
} RrsMaterialTag;

/* enum Fresnel, material.rs:124-129. */
typedef enum RrsFresnelKind { RRS_FRESNEL_DIELECTRIC = 0, RRS_FRESNEL_METALLIC = 1 } RrsFresnelKind;

/* One primitive, in the DFS leaf order of the reference tree (bvh.rs:391-415 visits
 * children left to right, so this order is the tie-break priority among equal t).
 * Geometry is carried in f64 exactly as the reference stores it; the library derives its
 * own fp32 records.
 *   sphere  : v[0]=radius^2 (Sphere stores radius2, geometry.rs:98-101), v[1..3]=centre
 *   plane   : v[0]=axis (RrsAxis), v[1]=umin v[2]=umax v[3]=vmin v[4]=vmax v[5]=pos
 *   triangle: v[0..2]=p1, v[3..5]=p2, v[6..8]=p3 */
typedef struct RrsPrim {
    uint32_t type;     /* RrsPrimType */
    uint32_t obj_id;   /* index of the object in the Vec<Object> given to Scene::new (lib.rs:227) */
    uint32_t material; /* index into RrsSceneDesc.materials */
    int32_t emission;  /* index into RrsSceneDesc.emissions, -1 = Emission::Dark */
    double v[9];
} RrsPrim;

/* Material parameters as the constructors take them (material.rs:595-716). */
typedef struct RrsMaterial {
    uint32_t tag;          /* RrsMaterialTag */
    uint32_t fresnel_kind; /* RrsFresnelKind; CookTorrance only (others are dielectric(ior)) */
    double color[3];
    double spec_color[3];  /* Plastic: spec_color; CookTorrance metallic: r0 */
    double alpha;          /* roughness alpha (the library squares it like CookTorrance::new) */
    double ior;
} RrsMaterial;

/* Emission::Emissive(strength, color), material.rs:1048-1084. */
typedef struct RrsEmission {
    double strength;
    double color[3];
} RrsEmission;

/* Child reference of a BVH node.  bit31 set: leaf run of primitives —
 * bits 0..27 = first primitive (index into prims), bits 28..30 = count-1 (1..4 prims,
 * bvh.rs:221-224,304-315: leaf groups hold <= 4 objects).  bit31 clear: index of another
 * RrsNode.  RRS_REF_EMPTY: no child (dead subtree, see `nodes`). */
#define RRS_REF_LEAF 0x80000000u
#define RRS_REF_EMPTY 0xFFFFFFFFu
#define RRS_MAKE_LEAF(first, count) (RRS_REF_LEAF | (((uint32_t)(count)-1u) << 28) | (uint32_t)(first))

/* 64-byte BVH node: one binary `BvhTree::Node` of the reference tree (bvh.rs:216-224) with
 * the boxes of BOTH children stored in the parent, so that one 2x256-bit fetch decides both
 * descents.  lo/hi are fp32, rounded outward from the f64 boxes of the reference.
 *  - child that is a `Node`          : box = that node's own bbox (geometry.rs:544-550);
 *  - child that is a bare `LeafNode` : the reference tests it whenever the parent is entered
 *    (it has no box); box = the primitive's bbox, or the parent's box if that is degenerate;
 *  - a `Node` whose own f64 box has zero extent on an axis can never be entered by the
 *    reference slab test (geometry.rs:474,491,508: tmax <= tmin) — it is stored as
 *    RRS_REF_EMPTY with an inverted box;
 *  - node 0 is a virtual root: child0 = the reference root (with its bbox), child1 empty.
 * NaN-free by construction. */
typedef struct RrsNode {
    float lo0[3], hi0[3];
    float lo1[3], hi1[3];
    uint32_t ref0, ref1;
    uint32_t flags; /* bit0: child0 has no box of its own in the reference (bare LeafNode); bit1: same for child1 */
    uint32_t pad;
} RrsNode;

/* f64 twin of RrsNode holding the reference's exact boxes; used only by the fp64
 * verification traversal (precision=64 in rrs_intersect). 128 bytes. */
typedef struct RrsNodeF64 {
    double lo0[3], hi0[3];
    double lo1[3], hi1[3];
    uint32_t ref0, ref1;
    uint32_t flags;
    uint32_t pad[5];
} RrsNodeF64;

typedef struct RrsSceneDesc {
    uint32_t abi_version; /* RRS_ABI_VERSION */
    uint32_t n_prims;
    const RrsPrim* prims;
    uint32_t n_nodes;
    const RrsNode* nodes;
    const RrsNodeF64* nodes_f64; /* may be NULL: precision=64 queries then fail with RRS_ERR_INVALID */
    uint32_t max_depth;          /* deepest chain of RrsNodes from node 0 (the host computes it; the library walks the
                                    tree itself and rejects a cycle, a node reached twice or a deeper chain) */
    uint32_t n_materials;
    const RrsMaterial* materials;
    uint32_t n_emissions;
    const RrsEmission* emissions;
    /* equirectangular environment, row-major RGB f32, already clipped by the caller as
     * rayrs/src/main.rs:43 does (Scene::background, lib.rs:254-285) */
    uint32_t hdri_width, hdri_height;
    const float* hdri_rgb;
    /* Scene::new z_near / z_far (lib.rs:227-245; main.rs:52 passes 1e-6, 1e6) */
    double t_min, t_max;
    uint32_t flags;        /* RRS_SCENE_* tuning switches, 0 = defaults */
    uint32_t refill_lanes; /* BVH traversal: idle lanes of a warp that trigger a fetch of new rays; 0 = library default */
} RrsSceneDesc;

/* RrsSceneDesc.flags (measurement switches: every one keeps the results identical) */
#define RRS_SCENE_NO_BRUTE 1u      /* scenes of <= 8 primitives: traverse the BVH instead of testing every primitive */
#define RRS_SCENE_NO_BRUTE_BOX 2u  /* ... keep the brute-force list but drop the box around its sphere group */
#define RRS_SCENE_NO_L2_PERSIST 4u /* never pin the node / primitive arrays in L2, and leave the device's persisting-L2 set-aside alone
                                      (by default a BVH render claims it and a small-scene render releases it) */

/* Derived camera fields exactly as Camera::new computes them (lib.rs:113-132), so that the
 * FOV quirk (z scaled by width/tan(fov/2)) stays on the host. */
typedef struct RrsCamera {
    double origin[3];
    double e_x[3];
    double e_y[3];
    double z_scaled[3];
    double width, height; /* film size in cm */
    uint32_t ppc;         /* pixels per cm */
    uint32_t x_pixels, y_pixels;
} RrsCamera;

typedef struct RrsRenderParams {
    uint32_t width, height;   /* must equal camera x_pixels / y_pixels */
    uint32_t spp;             /* samples per pixel rendered by THIS call */
    uint32_t sample_offset;   /* global index of the first sample (multi-GPU sample split) */
    uint32_t spp_total;       /* divisor for the mean written by rrs_render (0 => spp) */
    uint32_t max_bounces;     /* rayrs/src/main.rs:77 passes 50 */
    uint64_t seed;            /* key of the counter-based RNG */
    uint32_t queue_capacity;  /* rays in flight; 0 = library default */
    uint32_t flags;           /* RRS_FLAG_*, 0 = defaults */
} RrsRenderParams;

typedef struct RrsRay {
    double origin[3];
    double direction[3]; /* not normalised, like lib.rs:25-32 */
} RrsRay;

typedef struct RrsStats {
    uint64_t rays;            /* BVH queries (primary + every bounce) of the last render */
    uint64_t paths;           /* primary rays of the last render */
    uint64_t kernel_launches; /* kernels launched by the last render */
    uint64_t iterations;      /* wavefront iterations of the last render */
    uint64_t nan_pixels;      /* pixels with a NaN component (main.rs:81-83) */
    uint64_t negative_pixels; /* pixels with a negative component (main.rs:85-87) */
    double device_ms;         /* CUDA-event time of the last render (all kernels) */
    double extend_ms;         /* ... of its extend (traversal) launches, when profiling is on */
    double shade_ms;
    double generate_ms;
    uint64_t nodes_visited;   /* only with RRS_FLAG_COUNT_TRAVERSAL */
    uint64_t prims_tested;
    uint64_t kernel_form;     /* RRS_FORM_*: which render kernel the last render used */
    uint64_t census_mismatch_pixels; /* last resolve: pixels whose count of terminated paths != spp_total (the accumulator's
                                        .w lane counts them; 0 for a complete image — a built-in check of the queue
                                        bookkeeping and, on several GPUs, of the sample split + reduce) */
} RrsStats;

#define RRS_FORM_WAVEFRONT 0u /* fused persistent wavefront kernel, ray/hit queues in HBM (k_wavefront) */
#define RRS_FORM_SPLIT 1u     /* one generate/extend/shade launch per iteration (RRS_FLAG_SPLIT_KERNELS) */
#define RRS_FORM_PATHLOOP 2u  /* small scene: register-resident path loop, no queues (k_pathloop) */

#define RRS_FLAG_COUNT_TRAVERSAL 1u /* count nodes/primitives touched (slower; for the bytes/ray model) */
#define RRS_FLAG_TIME_PHASES 2u     /* split kernels only: CUDA-event time every phase launch */
#define RRS_FLAG_SPLIT_KERNELS 4u   /* one generate/extend/shade launch per wavefront iteration instead of the
                                       single fused persistent kernel (per-phase profiling) */
#define RRS_FLAG_FORCE_QUEUES 8u    /* use the queue-based wavefront kernel (the default; kept for A/B scripts) */
#define RRS_FLAG_NO_L2_WINDOW 32u    /* this render: no L2 access-policy window over the node / primitive arrays (A/B) */
#define RRS_FLAG_FORCE_PATHLOOP 16u /* small scenes (<= 8 primitives): use the register-resident path loop
                                       (k_pathloop) instead of the queued kernel (A/B measurements, tests) */
#define RRS_FLAG_ENV_SAMPLING 64u   /* next-event estimation of the environment map: at every Lambertian or CookTorrance
                                       vertex a direction is drawn from the map's importance-sampling table
                                       (rrs_env_sample) and traced as a shadow ray, combined with the BSDF-sampled
                                       continuation by multiple importance sampling (power heuristic).  The image
                                       converges to the same mean as without the flag — the reference's estimator,
                                       Russian roulette and quirks included — with less noise where the map's energy
                                       is concentrated (a sun).  Other materials (Plastic, the glass / refract
                                       variants, Reflect, NoReflect) and emission are shaded as without the flag.
                                       Runs the fused queued kernel (RRS_FORM_WAVEFRONT; never the path loop; not with
                                       RRS_FLAG_SPLIT_KERNELS) and doubles its ray queues. */

typedef struct RrsScene RrsScene;

/* Scene::new (lib.rs:227-245) device half: validates, converts and uploads.
 * An RrsScene carries mutable render state (ray queues, counters, staging buffers, statistics): one handle must
 * not be used from two threads or two streams at the same time.  Handles on different devices are independent. */
int rrs_scene_create(const RrsSceneDesc* desc, int device, RrsScene** out);
/* The same scene on n devices: validated and converted ONCE on the host, uploaded n times (the multi-GPU sample
 * split replicates the scene).  out[i] lives on devices[i]; on failure nothing is left allocated. */
int rrs_scene_create_multi(const RrsSceneDesc* desc, const int* devices, int n, RrsScene** out);
void rrs_scene_destroy(RrsScene* scene);

/* The render call (replaces rayrs/src/main.rs:61-94).  out_rgb: HOST buffer of
 * height*width*3 floats, row-major, row 0 = top (image.rs:140-165 layout); receives the
 * per-pixel MEAN radiance over spp_total samples (main.rs:89).  Synchronous. */
int rrs_render(RrsScene* scene, const RrsCamera* camera, const RrsRenderParams* params, float* out_rgb);

/* Same, but ACCUMULATES the per-pixel radiance SUM of this call's samples into a DEVICE
 * buffer of height*width float4 (rgb + sample count in .w), enqueued on `cuda_stream`
 * (a cudaStream_t; NULL = default stream).  ASYNCHRONOUS: the call returns once the work is enqueued (one
 * persistent kernel + a 128-byte counter read-back); rrs_stats / rrs_resolve / rrs_scene_destroy wait for it.
 * Only RRS_FLAG_SPLIT_KERNELS (per-phase profiling) polls the device and therefore blocks.
 * Used for the multi-GPU sample split: each GPU accumulates its slice, one reduce merges the buffers. */
int rrs_render_accumulate(RrsScene* scene, const RrsCamera* camera, const RrsRenderParams* params,
                          void* d_sum_rgba, void* cuda_stream);

/* ---- multi-GPU: samples of a pixel split over the GPUs of one box, ONE ncclReduce(sum) of the fp32 radiance
 * buffers (SURVEY.md 8e; the reference's seam is still the one render call, rayrs/src/main.rs:57-101).
 * NCCL is loaded at run time (dlopen "libnccl.so.2") the first time a communicator is made, so a single-GPU
 * host needs no NCCL; a missing library is RRS_ERR_COMM. */
typedef struct RrsComm RrsComm;
typedef struct RrsUniqueId { char bytes[128]; } RrsUniqueId; /* ncclUniqueId */

/* (first global sample, number of samples) of `rank` among `world`: contiguous, disjoint, covering [0, spp);
 * the first spp % world ranks take one extra sample. */
int rrs_sample_range(uint32_t rank, uint32_t world, uint32_t spp, uint32_t* first, uint32_t* count);

/* one process driving n devices (ncclCommInitAll): local rank i = global rank i on devices[i] */
int rrs_comm_init_all(const int* devices, int n, RrsComm** out);
/* one process per device: rank 0 makes the id, the host passes it to the other ranks by its own means
 * (a file, MPI, torch.distributed ...), every rank then joins (ncclCommInitRank; collective) */
int rrs_comm_unique_id(RrsUniqueId* out);
int rrs_comm_init_rank(const RrsUniqueId* id, int world, int rank, int device, RrsComm** out);
void rrs_comm_destroy(RrsComm* comm);

/* The render call on several GPUs.  scenes[i] (i < n_local) is the scene on the i-th device of `comm`
 * (n_local = n for rrs_comm_init_all, 1 for rrs_comm_init_rank; collective across processes in the second case).
 * params->spp is the TOTAL sample count of the image (sample_offset = first global sample, normally 0); every
 * global rank renders rrs_sample_range(rank, world, spp) into its own radiance buffer, the buffers are summed
 * on global rank 0 by one ncclReduce, and rank 0 divides by spp and counts NaN / negative pixels.
 * out_rgb (height*width*3 floats; host memory, or device memory on rank 0's GPU when out_is_device) is written
 * by the process that holds global rank 0 and ignored elsewhere (may be NULL there).
 * cuda_streams: n_local cudaStream_t to enqueue on, or NULL for the library's own per-device streams.
 * Returns after the image is complete on rank 0 (other ranks: after their part is enqueued and the
 * reduce has been issued; rrs_stats waits).  The RNG is keyed by the global sample index, so the
 * image is independent of the number of GPUs up to fp32 summation order. */
int rrs_render_multi(RrsScene* const* scenes, int n_local, RrsComm* comm, const RrsCamera* camera,
                     const RrsRenderParams* params, float* out_rgb, int out_is_device, void* const* cuda_streams);

/* d_sum_rgba (device, float4 per pixel) -> out (device or host per `out_is_device`) mean
 * RGB f32, dividing by spp_total, and counting NaN / negative pixels into the stats. */
int rrs_resolve(RrsScene* scene, const void* d_sum_rgba, uint32_t width, uint32_t height, uint32_t spp_total,
                float* out_rgb, int out_is_device, void* cuda_stream);

/* Output stage on the device — Image::to_raw_bytes (image.rs:193-222) fused with the division by
 * spp_total: d_sum_rgba (device, float4 per pixel) -> out_rgb8 (device or host per `out_is_device`),
 * 3 bytes per pixel = (255.99 * clip(mean, 0, 1)^gamma) as u8, evaluated in f64 like the reference
 * (a NaN component clips to 1, as f64::min/max do).  census3, if not NULL, receives the three counters
 * the reference prints: [clamped (> 1), NaN, negative] pixels.  The HDR export of main.rs:113-121
 * (Image::pixels_f32, image.rs:224-229) is what rrs_resolve already returns.  Synchronous. */
int rrs_to_raw_bytes(RrsScene* scene, const void* d_sum_rgba, uint32_t width, uint32_t height, uint32_t spp_total,
                     double gamma, uint8_t* out_rgb8, int out_is_device, void* cuda_stream, uint64_t* census3);

/* Closest hit for a batch of rays — Bvh::intersect (bvh.rs:212-214) with the scene's
 * (t_min, t_max).  obj_id[i] = RrsPrim.obj_id of the hit or -1; t[i] = distance or +inf.
 * precision 32: the production fp32 traversal (ordered, t-pruned).
 * precision 64: fp64 literal traversal (reference visiting order, no pruning, no FMA)
 *               for verification. */
int rrs_intersect(RrsScene* scene, const RrsRay* rays, size_t n, int32_t* obj_id, double* t, int precision);

/* Material::evaluate (material.rs:91-109, pdf=None) for a batch: normal_view = n x 6 doubles
 * (unit normal, unit view), u = n x 3 uniforms in call order; out = n x 7 floats
 * [scatter flag, color rgb, direction xyz].  Parity probe for the shading kernels.  The kernels carry two
 * forms of the function (shared stages for mixed warps, one arm per variant for the small-scene path loop);
 * `material | RRS_MATERIAL_FORM_CASES` probes the second. */
#define RRS_MATERIAL_FORM_CASES 0x80000000u
int rrs_material_evaluate(RrsScene* scene, uint32_t material, const double* normal_view, const double* u,
                          size_t n, float* out);

/* Material::evaluate WITH a caller's pdf — the reference's dormant next-event-estimation hook.  material.rs:91-109 hands
 * `pdf: Option<Pdf>` to every Bsdf::scatter; the one arm that looks at it is LambertianDiffuse::scatter (material.rs:259-281),
 * reached directly or as Plastic's diffuse lobe (:588): it samples and weights the lobe with
 * Pdf::Mix(MixKind::Constant(0.5), pdf, Pdf::Cosine) (generate :1028-1034, value :951-959).  Here pdf =
 * Pdf::Hittable(&geometry of `light`) (value :943-950, generate :1027; Hittable::area / sample geometry.rs:138-152,
 * 284-299,381-387), `light` being the caller's f64 record of the sampled primitive (any entry of RrsSceneDesc.prims).
 *   pos_normal_view  n x 9 doubles: shaded position, unit normal, unit view
 *   u                n x 4 uniforms in call order (Lambertian: side of the mix, then the two draws of the chosen
 *                    generator; Plastic: its lobe choice first)
 *   out              n x 7 doubles [scatter flag, color rgb, direction xyz]
 * radiance() passes None (lib.rs:532): no render reaches this, the reference's or ours.  The hook is therefore
 * evaluated in f64 with the reference's operation order (held to the oracle at rounding level); materials and lobes
 * that ignore the pdf return what rrs_material_evaluate returns (fp32 production shading, draws u[0..2]).
 * Reference quirks kept as written: Sphere::sample is not uniform (its own FIXME), Triangle::sample returns the
 * origin, Pdf::Hittable::value divides by the cosine at the shaded point. */
int rrs_material_evaluate_pdf(RrsScene* scene, uint32_t material, const RrsPrim* light, const double* pos_normal_view,
                              const double* u, size_t n, double* out);

/* Scene::background (lib.rs:254-285) for a batch of directions (n x 3 doubles) -> n x 3 floats. */
int rrs_background(RrsScene* scene, const double* dirs, size_t n, float* out);

/* Parity probes of RRS_FLAG_ENV_SAMPLING's environment sampler.  rrs_env_sample: u = n x 2 uniforms in [0, 1) ->
 * dir_pdf = n x 4 [unit direction xyz, solid-angle density] of the direction the render draws for them (each
 * uniform's top 24 bits pick the cell of the table, the rest place the direction inside it).  Fails with
 * RRS_ERR_INVALID on a black map.  rrs_env_pdf: dirs = n x 3 (need not be unit) -> pdf = n densities, exactly as the
 * render evaluates them; 0 where the map is black.  The table is built once per scene by rrs_scene_create over the
 * (w-1) x (h-1) cells between texel centres (4 bytes per cell + 8 per row of device memory). */
int rrs_env_sample(RrsScene* scene, const double* u, size_t n, double* dir_pdf);
int rrs_env_pdf(RrsScene* scene, const double* dirs, size_t n, double* pdf);

/* The uniforms the device RNG hands to (pixel, sample, slot): 4 floats. */
int rrs_rng_uniforms(RrsScene* scene, uint64_t seed, uint32_t pixel, uint32_t sample, uint32_t slot, float* out4);

/* ---- BvhTree::build_sah / build_midpoint (bvh.rs:227-389) on the device: the SAME tree as the reference's recursive
 * build — same boxes bit for bit, same split indices, same primitive order — as a level-synchronous sweep (stable
 * radix sort per level, segmented prefix / suffix box scans, the calculate_sah sweep over the splits the threshold
 * loop reaches).  Scene setup for hosts whose own build is the bottleneck (4M triangles: seconds on the host);
 * the host flattens the returned tree into RrsNode / RrsPrim exactly as it would its own.
 *   boxes      n x 6 doubles, one object each: xmin, xmax, ymin, ymax, zmin, zmax (Hittable::bbox)
 *   heuristic  0 = BvhHeuristic::Midpoint, 1 = BvhHeuristic::Sah { splits }
 *   prim_order n entries out: object indices in DFS leaf order
 *   nodes      capacity 2 n + 2 out: node 0 is the root; kind 0 = Node with two children (indices into nodes),
 *              1 = Node holding <= 4 LeafNodes (objects prim_order[first .. first + count)), 2 = bare LeafNode
 *              (object prim_order[first]; box = the object's own)
 *   seconds    device time of the build (may be NULL) */
typedef struct RrsBuildNode {
    double box[6];
    int32_t child[2];
    uint32_t first, count;
    uint32_t kind, pad;
} RrsBuildNode;
int rrs_bvh_build(const double* boxes, uint32_t n, uint32_t heuristic, uint32_t splits, int device, uint32_t* prim_order,
                  RrsBuildNode* nodes, uint32_t* n_nodes, double* seconds);

int rrs_stats(RrsScene* scene, RrsStats* out);
const char* rrs_last_error(void);
int rrs_abi_version(void);
/* number of usable sm_100 devices (0 => every device call fails with RRS_ERR_NO_DEVICE) */
int rrs_device_count(void);

#ifdef __cplusplus
}
#endif
#endif /* RAYRS_B200_H */
