/* lasgun_b200.h — C ABI of the B200 render path for nfrasser/lasgun.
 *
 * The reference has no FFI (SURVEY.md D4); its drop-in surface is the Rust public API
 *   lasgun::capture(&Scene, &mut Film)                      src/lib.rs:55
 *   lasgun::capture_subset(k, n, &Accel, &mut impl Img)     src/lib.rs:110
 *   lasgun::Accel::from(&Scene)                             src/lib.rs:42, src/accelerators/bvh.rs:135
 * A Rust `capture` shim builds its BVHAccel as today, flattens the (crate-private) fields
 * `nodes`, `order`, `primitives` (bvh.rs:48-69) into the arrays of `lgb_scene_desc`, and calls
 * the functions below (INTEGRATION.md shows the binding).  Everything from camera ray generation
 * (camera.rs:113-146) through traversal (bvh.rs:461-522), primitive intersection
 * (sphere.rs:79, cuboid.rs:55, triangle.rs:161), shading (integrate.rs:23-80) and film
 * quantisation (img.rs:56-67) then runs in sm_100a CUDA kernels.
 *
 * Conventions: every function returns LGB_OK (0) or a negative lgb_status; nothing aborts or
 * unwinds across this boundary.  Host arrays passed in are borrowed for the duration of the
 * call only.  One capture at a time per context.  One context drives one GPU; multi-GPU
 * renders use one context per GPU (one process per GPU) and the tile-rank arguments.
 */
#ifndef LASGUN_B200_H
#define LASGUN_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LGB_ABI_VERSION 5

typedef enum lgb_status {
    LGB_OK = 0,
    LGB_ERR_INVALID = -1,      /* bad argument / malformed scene description */
    LGB_ERR_CUDA = -2,         /* CUDA runtime failure (see lgb_last_error) */
    LGB_ERR_UNSUPPORTED = -3,  /* feature outside the hot path (material, transform, depth > 64) */
    LGB_ERR_NOMEM = -4,
    LGB_ERR_NO_DEVICE = -5     /* no sm_100-class GPU: there is NO CPU fallback */
} lgb_status;

typedef struct lgb_ctx lgb_ctx;
typedef struct lgb_scene lgb_scene;

/* Primitive reference stored in a BVH leaf: (type << 30) | index into that type's array.
 * Leaf order is the reference's `order[]` already applied (bvh.rs:484). */
enum { LGB_PRIM_SPHERE = 0, LGB_PRIM_CUBOID = 1, LGB_PRIM_TRIANGLE = 2, LGB_PRIM_INSTANCE = 3 };
#define LGB_PRIM_REF(type, index) (((uint32_t)(type) << 30) | (uint32_t)(index))
#define LGB_MISS 0xFFFFFFFFu

/* Flattened BVH node, 32 bytes, pre-order as flatten_bvh_tree (bvh.rs:430-453): the left child of
 * an interior node is index + 1.  Boxes must contain the reference's f64 box (round outward).
 *   interior: a = index of the second child, b = split axis (0..2)
 *   leaf:     a = first entry in prim_refs, b = LGB_LEAF_FLAG | count
 * Child indices and instance roots are absolute indices into the one `nodes` array. */
#define LGB_LEAF_FLAG 0x80000000u
typedef struct lgb_node {
    float lo[3]; uint32_t a;
    float hi[3]; uint32_t b;
} lgb_node;

typedef struct lgb_sphere {          /* Sphere, src/shape/sphere.rs:12-16 */
    double center[3]; double radius;
} lgb_sphere;

typedef struct lgb_cuboid {          /* Cuboid bounds, src/shape/cuboid.rs:12-30 */
    double min[3]; double max[3];
} lgb_cuboid;

typedef struct lgb_triangle {        /* the three f32 OBJ positions a Triangle reads, triangle.rs:40-55 */
    float p0[3]; float p1[3]; float p2[3];
} lgb_triangle;

typedef struct lgb_tri_normals {     /* per-vertex f32 normals, triangle.rs:58-76 */
    float n0[3]; float n1[3]; float n2[3];
} lgb_tri_normals;

/* Nested BVH used as a primitive (bvh.rs:141-162), with the Transform3 of its aggregate (scene/node.rs:86-115,
 * space/transform.rs:48-197).  The ray is taken into the level's space with `minv` (transform.rs:279-283: t is
 * preserved because d is not renormalised) and the hit record comes back with `m` (transform.rs:243-264), then
 * swap_backface (bvh.rs:518).  Matrices are cgmath Matrix4<f64>, column-major: element [c][r] at index 4*c + r.
 * They must be affine (row 3 = 0 0 0 1); `identity` = 1 promises that both are the identity. */
typedef struct lgb_instance {
    uint32_t root_node;              /* absolute index of the child BVH's node 0 */
    uint32_t identity;
    uint32_t swap_backface;
    uint32_t reserved;
    double m[16], minv[16];
} lgb_instance;

/* `Material` (material/mod.rs:4-46), one record for the five variants:
 *   LGB_MAT_MATTE    kd, roughness = sigma in degrees, already clamped to [0, 90] (matte.rs:15); sigma == 0: Lambertian only
 *   LGB_MAT_PLASTIC  kd, ks, roughness (plastic.rs)
 *   LGB_MAT_METAL    kd = eta, ks = k, roughness = u_roughness, roughness_v = v_roughness (metal.rs)
 *   LGB_MAT_GLASS    kd = kr, ks = kt, roughness = eta (glass.rs; Material::glass passes no microfacet roughness, mod.rs:36-41)
 *   LGB_MAT_MIRROR   kd = kr (mirror.rs)
 * Glass and mirror scatter through the Whitted recursion of integrate.rs:69-132, to depth lgb_scene_desc.recursion. */
enum { LGB_MAT_MATTE = 0, LGB_MAT_PLASTIC = 1, LGB_MAT_METAL = 2, LGB_MAT_GLASS = 3, LGB_MAT_MIRROR = 4 };
typedef struct lgb_material {
    double kd[3]; double roughness;
    double ks[3]; double roughness_v;
    uint32_t kind; uint32_t reserved;
} lgb_material;

typedef struct lgb_light {           /* PointLight, src/light/point.rs:14-18 */
    double position[3]; double intensity[3]; double falloff[3];
} lgb_light;

typedef struct lgb_camera {          /* Camera after look_at, src/camera.rs:6-38 */
    double origin[3], view[3], up[3], aux[3];
    double image_plane_height;       /* camera.rs:93, :158-164 */
    double pixel_separation;         /* 0 perspective, 1 orthographic (camera.rs:168-173) */
    double sample_distance;          /* Supersampling::distance = 1 / root (camera.rs:189-193) */
    uint32_t supersampling_root;     /* samples per pixel = root * root */
    uint32_t reserved;
} lgb_camera;

/* Lazy reference tree.  The device traverses its own BVH; the caller's (reference) tree is consulted for ONE thing:
 * the order in which the reference tests primitives, which decides exact-t ties (see below).  Most frames contain no
 * such tie.  A caller may therefore leave `nodes` NULL and give a callback instead: it is invoked -- from the thread
 * that calls lgb_capture*, at most once per scene -- only if a closest-hit ray meets two primitives at bit-identical t;
 * the affected rays are then re-traced with the order known.  The reference BVH build (the larger part of the host
 * time of `capture`) is skipped otherwise.  Lazy scenes must not contain transformed instances (their spaces are
 * derived from the tree) and need `bounds_lo/hi`: a world box containing every primitive (the reference root box).
 * The primitive arrays of the desc must stay valid until the scene is destroyed. */
typedef struct lgb_reference_tree {
    const lgb_node* nodes;           uint64_t n_nodes;
    const uint32_t* prim_refs;       uint64_t n_prim_refs;
    const lgb_instance* instances;   uint64_t n_instances;
} lgb_reference_tree;
typedef int (*lgb_reference_tree_fn)(void* user, lgb_reference_tree* out);   /* 0 = ok; arrays stay owned by the caller */

typedef struct lgb_scene_desc {
    uint32_t abi_version;            /* LGB_ABI_VERSION */
    uint32_t flags;                  /* LGB_SCENE_* */
    const lgb_node* nodes;           uint64_t n_nodes;       /* node 0 = root of the top-level BVH */
    const uint32_t* prim_refs;       uint64_t n_prim_refs;
    const lgb_sphere* spheres;       uint64_t n_spheres;
    const uint32_t* sphere_material; const uint32_t* sphere_id;      /* n_spheres each */
    const lgb_cuboid* cuboids;       uint64_t n_cuboids;
    const uint32_t* cuboid_material; const uint32_t* cuboid_id;      /* n_cuboids each */
    const lgb_triangle* triangles;   uint64_t n_triangles;
    const uint32_t* triangle_material; const uint32_t* triangle_id;  /* n_triangles each */
    const lgb_tri_normals* tri_normals;  /* NULL or n_triangles entries (mesh has normals and smoothing is on) */
    const uint8_t* tri_has_normals;      /* NULL or n_triangles flags (meshes may differ) */
    const lgb_instance* instances;   uint64_t n_instances;
    lgb_instance root;               /* transform / swap_backface of the root aggregate itself (root_node = 0) */
    const lgb_material* materials;   uint64_t n_materials;
    const lgb_light* lights;         uint64_t n_lights;      /* at most LGB_MAX_LIGHTS */
    lgb_camera camera;
    double ambient[3];                                       /* scene.rs:22 */
    double bg_inner[3], bg_outer[3], bg_scale;               /* material/background.rs:6-10 */
    uint32_t recursion;                                      /* scene.recursion (scene.rs:60, default 3): Whitted depth, at most 12 */
    uint32_t expected_film_pixels;                           /* hint, 0 = unknown: w * h of the film `capture` is about to fill (lib.rs:55 knows it).
                                                              * With it lgb_scene_create can tell whether the frame will walk the device BVH at all
                                                              * and leave the tree unbuilt otherwise (LGB_OPT_LAZY_BVH); results never depend on it. */
    lgb_reference_tree_fn reference_tree;                    /* lazy mode (nodes == NULL), else NULL */
    void* reference_tree_user;
    double bounds_lo[3], bounds_hi[3];                       /* lazy mode: world box of all primitives */
} lgb_scene_desc;

#define LGB_MAX_LIGHTS 32
/* The caller's tree is the REFERENCE tree.  lgb_scene_create uses it (a) to validate the scene and bound
 * the traversal stack as the reference would, and (b) to record, per ray-direction octant, the order in
 * which the reference tests primitives, which is how exact-t ties are resolved (first tested wins,
 * sphere.rs:86 / cuboid.rs:95 / triangle.rs:251).  The device traverses its own SAH BVH over the same
 * primitives; results are the reference's for any such BVH.  Pass the tree exactly as the reference built
 * it (leaves of up to 254 primitives, bvh.rs:289): re-splitting its leaves would change the test order. */

typedef struct lgb_stats {
    uint64_t primary_rays;           /* w * h * spp rendered by this call */
    uint64_t primary_hits;
    uint64_t shadow_rays;            /* reference semantics: lights * primary_hits (integrate.rs:47-50) */
    uint64_t shadow_rays_traced;     /* shadow rays the device resolved (lights that can contribute, bsdf.rs:75) */
    uint64_t shadow_occluded;
    uint64_t shadow_cache_hits;      /* of those: blocked by the occluder of the pixel's anchor sample, no traversal */
    /* Work counters, filled only by lgb_capture_aov or with LGB_OPT_COUNT_WORK (slower kernel variant);
     * index 0 sphere, 1 cuboid, 2 triangle. */
    uint64_t exact_tests[3];         /* f64 reference-arithmetic primitive tests executed */
    uint64_t filter_tests[3];        /* conservative f32 primitive filter tests executed */
    uint64_t node_tests;             /* node fetches; each one tests two child boxes */
    uint64_t primary_node_tests;     /* the share of the closest-hit (primary ray) kernel in the three counters above */
    uint64_t primary_exact_tests[3];
    uint64_t primary_filter_tests[3];
    /* device time of each phase of the frame (CUDA events on the launch stream): 0 primary rays, 1 hit setup +
     * shadow queues, 2 anchor shadow rays, 3 cached-occluder test + remaining shadow rays, 4 shade, 5 resolve */
    float kernel_ms[6];
    float render_ms;                 /* device time of the render + resolve kernels */
    float total_ms;                  /* device time incl. film copy back to the host */
    uint32_t kernel_launches;
    uint32_t stack_overflow;         /* 1 if a ray exceeded the 64-entry stack (bvh.rs:469) */
    uint32_t beams;                  /* 1 if the primary (and shadow) rays went through pixel beams (LGB_OPT_BEAMS) */
    uint32_t tie_retraces;           /* lazy reference tree: sample slots re-traced because of an exact-t tie (this call) */
    uint64_t secondary_rays;         /* rays below specular hits (reflected, transmitted and their shadow rays), integrate.rs:69-132 */
    uint32_t bands;                  /* passes the frame was rendered in (per-sample buffers are sized by LGB_OPT_WAVE_BUDGET_MB) */
    uint32_t reserved;
} lgb_stats;

/* Shared film (multi-GPU, one process per GPU): rank 0 allocates the film and hands the 64-byte handle to the other
 * processes; they map it and pass the mapped pointer as `d_film` of lgb_capture_device, so their resolve stage stores
 * its uchar4 pixels straight into rank 0's HBM over NVLink -- the gather IS the kernel's stores, there is no collective
 * on the data path (SURVEY 8e).  The tiles of the ranks are disjoint; a barrier after the captures completes the frame. */
#define LGB_IPC_HANDLE_BYTES 64
int lgb_film_alloc_shared(lgb_ctx* ctx, uint64_t bytes, void** d_film, uint8_t handle_out[LGB_IPC_HANDLE_BYTES]);
int lgb_film_open_shared(lgb_ctx* ctx, const uint8_t handle[LGB_IPC_HANDLE_BYTES], void** d_film);
int lgb_film_release_shared(lgb_ctx* ctx, void* d_film, int owner);   /* owner != 0: cudaFree, else cudaIpcCloseMemHandle */
/* End-of-frame flags for a shared film: words of the SAME shared allocation (allocate a little more than w*h*4).  lgb_film_signal
 * queues, behind the caller's kernels on `stream`, a system-fenced store of `value` into *d_flag (own or peer memory);
 * lgb_film_wait queues a kernel that returns once the n words d_flags[(first + i) * stride_bytes / 4] have all reached `value`
 * (values only grow; it gives up after minutes instead of hanging the GPU).  A rank signals its word when its tiles are stored,
 * rank 0 waits for all of them: the frame barrier costs two microsecond kernels and no collective (lasgun_b200/multi.py). */
int lgb_film_signal(lgb_ctx* ctx, void* d_flag, uint32_t value, void* stream);
int lgb_film_wait(lgb_ctx* ctx, const void* d_flags, uint32_t first, uint32_t n, uint32_t stride_bytes, uint32_t value, void* stream);

/* Device / context --------------------------------------------------------------------- */
int lgb_device_count(void);
int lgb_init(int device, lgb_ctx** out);
/* A device group in ONE process: the analogue of the reference's worker threads (src/lib.rs:55-104 spawns num_cpus of them
 * inside one blocking `capture`).  devices[0] leads: scenes are built there and their arena is copied to the others over
 * NVLink (not rebuilt); lgb_capture and lgb_capture_device(tile_ranks = 1) then split the macro tiles over all listed
 * devices, each one's kernels store their pixels straight into the leader's film (peer access is required and checked here),
 * and the call returns when every device is done.  Every other entry point runs on the leader alone.  The returned context
 * is used exactly like a single-device one; lgb_shutdown closes the whole group. */
int lgb_init_devices(int n_devices, const int* devices, lgb_ctx** out);
int lgb_context_devices(const lgb_ctx* ctx);       /* devices a context renders on (1 for lgb_init) */
void lgb_shutdown(lgb_ctx* ctx);
#define LGB_OPT_COUNT_WORK 1        /* value != 0: captures also fill the work counters of lgb_stats */
#define LGB_OPT_SIDE_STREAMS 4      /* 1 (default): the shadow-ray kernels of different lights overlap on a side stream; 0: one stream */
#define LGB_OPT_WHITTED 3           /* glass / mirror ray trees: 1 (default) level-by-level wavefront on the frame's own kernels, 0 one thread per tree */
#define LGB_OPT_BEAMS 2             /* pixel beams: at >= 4 samples per pixel the primary rays of a pixel share ONE bundle traversal
                                     * (k_beam) and then test only the primitives it listed; likewise the shadow rays of a pixel
                                     * whose centre sample is unoccluded (k_sbeam, from the light).  Same results.  1 on, 0 off,
                                     * -1 (default) automatic: on for >= 8 samples per pixel and a BVH of >= 1024 nodes.
                                     * env LGB_BEAMS presets it. */
#define LGB_OPT_LIGHT_GRIDS 5       /* shadow rays through per-light cube-map grids of primitive lists instead of the BVH (csrc/lgb_grid.cu;
                                     * scenes without transformed aggregates).  Same occlusion bits.  1 on, 0 off, -1 (default)
                                     * automatic: device BVH of >= 1024 nodes and at most 8 lights.  Read at lgb_scene_create.
                                     * env LGB_LIGHT_GRIDS presets it. */
#define LGB_OPT_CAMERA_GRID 6       /* primary rays of a perspective camera through a grid of pixel tiles, each listing the primitives its
                                     * samples can see (csrc/lgb_grid.cu), instead of the BVH / pixel beams.  Same hits.  1 on, 0 off,
                                     * -1 (default) automatic.  Built at the first capture of a film size and kept with the scene.
                                     * env LGB_CAMERA_GRID presets it. */
#define LGB_OPT_WAVE_BUDGET_MB 7    /* memory (MB, default 16384) the per-sample wavefront buffers of one capture may take: a frame that needs more
                                     * is rendered in bands of macro tiles on the same buffers (any frame size in bounded memory).
                                     * env LGB_WAVE_BUDGET_MB presets it. */
#define LGB_OPT_LAZY_BVH 8          /* 1 / -1 (default): a plastic scene large enough for the device-side builder is created WITHOUT its BVH when light
                                     * grids will serve its shadow rays; the tree is built (6-8 ms for 0.6-1 M primitives) only if an entry point
                                     * walks one (a frame the camera grid does not serve, lgb_trace_rays, lgb_scene_verify, lgb_scene_export).
                                     * 0: always at lgb_scene_create.  env LGB_LAZY_BVH presets it. */
int lgb_set_option(lgb_ctx* ctx, int option, int value);
const char* lgb_last_error(lgb_ctx* ctx);          /* ctx may be NULL: last error of lgb_init */
const char* lgb_status_string(int status);

/* Scene: copies the caller's flat arrays to the device (replaces the data a BVHAccel owns). */
int lgb_scene_create(lgb_ctx* ctx, const lgb_scene_desc* desc, lgb_scene** out);
void lgb_scene_destroy(lgb_scene* scene);
uint64_t lgb_scene_device_bytes(const lgb_scene* scene);
/* Replication across GPUs (one process per GPU): the device scene is ONE relocatable arena plus a small layout
 * record.  The rank that built it exports both; the others receive the arena bytes over NVLink (NCCL broadcast, or
 * a peer copy) into memory they own and import it -- the BVH is built once, not once per GPU.
 * The imported scene borrows `arena_dev`: keep it alive until lgb_scene_destroy. */
uint64_t lgb_scene_layout_bytes(void);
int lgb_scene_export(const lgb_scene* scene, void* layout_out, uint64_t layout_bytes, void** arena_dev, uint64_t* arena_bytes);
int lgb_scene_import(lgb_ctx* ctx, const void* layout, uint64_t layout_bytes, void* arena_dev, lgb_scene** out);
double lgb_scene_build_ms(const lgb_scene* scene);       /* host time spent building the device BVH */
uint32_t lgb_scene_node_count(const lgb_scene* scene);   /* nodes of the device BVH */

/* Host-only probe (no GPU needed): runs the same validation, rank-table and device-BVH construction as
 * lgb_scene_create and checks the result (every primitive in exactly one leaf, boxes nested). */
typedef struct lgb_build_info {
    uint32_t nodes, max_depth, leaves, max_leaf;
    uint32_t prims, ranks_ok, boxes_ok, reserved;
    double build_ms, rank_ms, sah_cost;
} lgb_build_info;
int lgb_build_probe(const lgb_scene_desc* desc, lgb_build_info* out);
/* Reads the resident device BVH of a single-space scene back and checks it: every primitive in exactly one leaf
 * (canonical ids 0 .. prims-1 seen once), every primitive inside its leaf box, leaves <= 4 primitives.  Fills
 * nodes / max_depth / leaves / max_leaf / prims / boxes_ok / sah_cost; ranks_ok = 1 if the tree was built on the device. */
int lgb_scene_verify(lgb_ctx* ctx, const lgb_scene* scene, lgb_build_info* out);

/* capture (src/lib.rs:55): blocking; fills caller-owned row-major RGBA8, w*h*4 bytes (host). */
int lgb_capture(lgb_ctx* ctx, lgb_scene* scene, uint32_t w, uint32_t h, uint8_t* rgba_out, lgb_stats* stats);

/* capture_subset (src/lib.rs:110): pixels k, k+n, k+2n, ... of the row-major film only; all other
 * bytes of rgba_inout (host) are left untouched. */
int lgb_capture_subset(lgb_ctx* ctx, lgb_scene* scene, uint32_t k, uint32_t n, uint32_t w, uint32_t h,
                       uint8_t* rgba_inout, lgb_stats* stats);

/* Debug / parity: full-frame capture that also returns, per sample (index (y*w + x)*spp + s, sample
 * order of camera.rs:137-145), the canonical id of the closest-hit primitive (LGB_MISS if none), its
 * f64 ray parameter t (+inf if none), a bit mask of occluded lights and the sample's radiance (3 doubles: `li`,
 * integrate.rs:23, before the weighted sum of integrate.rs:16-20).  Any pointer may be NULL. */
int lgb_capture_aov(lgb_ctx* ctx, lgb_scene* scene, uint32_t w, uint32_t h, uint8_t* rgba_out,
                    uint32_t* prim_id, double* t, uint32_t* occluded, double* li, lgb_stats* stats);

/* Device-resident capture for benchmarks and multi-GPU: renders the macro-tiles owned by
 * `tile_rank` of `tile_ranks` (all tiles when tile_ranks == 1) into `d_film`, a DEVICE pointer to a
 * full w*h*4 row-major film that may live on a peer GPU.  Asynchronous on `stream` (a cudaStream_t,
 * NULL = the context's stream) unless `stats` is non-NULL, in which case it synchronises. */
int lgb_capture_device(lgb_ctx* ctx, lgb_scene* scene, uint32_t w, uint32_t h, uint32_t tile_rank,
                       uint32_t tile_ranks, void* d_film, void* stream, lgb_stats* stats);

/* Per-kernel timing of one frame (bench / roofline): the frame of lgb_capture_device (all tiles) with a pair of CUDA events around
 * EVERY kernel launch, all launches on one stream (the shadow chains of different lights do not overlap in this call), and, with
 * LGB_OPT_COUNT_WORK set, each launch's share of the work counters.  Entries come in launch order; *n_out is the number of
 * launches (entries beyond `cap` are dropped).  d_film: device film or NULL (the context's own).  Synchronises. */
typedef struct lgb_kernel_time {
    char name[40];                   /* kernel, "[light l]" appended for the per-light launches */
    float ms;
    uint32_t reserved;
    uint64_t node_tests;             /* work counters of this launch alone (zero unless LGB_OPT_COUNT_WORK): see lgb_stats */
    uint64_t filter_tests[3], exact_tests[3];
    uint64_t primary_rays, primary_hits, shadow_rays, shadow_occluded;
} lgb_kernel_time;
int lgb_capture_profile(lgb_ctx* ctx, lgb_scene* scene, uint32_t w, uint32_t h, void* d_film,
                        lgb_kernel_time* out, uint32_t cap, uint32_t* n_out, lgb_stats* stats);

/* Trace caller-supplied rays (o[3], d[3] f64 each) through the scene: closest-hit id, t and the world-space
 * RayIntersection::ng() / ns() (surface.rs:107-118; any output pointer may be NULL).
 * The f32 error bound of the traversal is derived from the world box of the scene and its camera (the reference root box,
 * through the root transform, united with the camera origin).  The f32 culling ray of an origin outside that box starts where
 * the ray enters it (grown by 1/64 of its extent), and a direction with max |d_k| outside [2^-40, 2^40] is traced scaled by
 * an exact power of two; the exact f64 tests give the reference's t either way.  Precondition: every origin lies within one
 * box extent of that box (so no coordinate is NaN or infinite); otherwise the whole batch is refused with LGB_ERR_UNSUPPORTED
 * and lgb_last_error names the box.
 * Used by the known-answer tests (tests/test_gpu_parity.py) and the random-ray parity tests (tests/test_trace_rays.py). */
int lgb_trace_rays(lgb_ctx* ctx, lgb_scene* scene, const double* rays_od, uint64_t n_rays,
                   uint32_t* prim_id, double* t, double* ng, double* ns);

/* Debug / parity: the reciprocal and reciprocal square root the shading kernel uses in place of IEEE division / sqrt
 * (MUFU seed + one third-order refinement, csrc/lgb_math.cuh) evaluated on caller-supplied positive normal doubles;
 * the tests bound their relative error (a few 1e-16).  They only colour: no hit, shadow or sign decision goes through them. */
int lgb_debug_fastmath(lgb_ctx* ctx, const double* x, uint64_t n, double* rcp_out, double* rsqrt_out);

/* Measured device ceilings used for roofline reporting (bench only). */
int lgb_measure_l2_read_gbs(lgb_ctx* ctx, uint64_t bytes, int iters, double* gbs_out);
int lgb_measure_fp32_gops(lgb_ctx* ctx, int iters, double* glaneops_out);
int lgb_measure_fp64_gops(lgb_ctx* ctx, int iters, double* glaneops_out);

#ifdef __cplusplus
}
#endif
#endif /* LASGUN_B200_H */
