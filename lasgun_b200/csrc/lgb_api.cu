// C-ABI glue (include/lasgun_b200.h): context, scene upload, capture entry points.
// No torch types, no CPU fallback: without an sm_100-class device lgb_init fails.
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <vector>

#include <thread>

#include "lgb_build.hpp"
#include "lgb_gpubuild.cuh"
#include "lgb_grid.cuh"
#include "lgb_parallel.hpp"
#include "lgb_types.cuh"

namespace lgb {
constexpr int kRenderEvents = 7;
cudaError_t launch_render(const DevScene&, const DevCamera&, const DevShade&, const DevWork&, const DevOut&, const DevWave&, bool stats, bool all_shadows, int sms, cudaStream_t, cudaEvent_t* ev, int part, const SideStreams* side, KernelLog* klog, ShadeChunks* chunks = nullptr);
bool render_fused(uint32_t spp);
bool surface_fused(const DevScene&, const DevWork&, const DevOut&, bool all_shadows);
bool setup_fused(const DevScene&, const DevWork&, const DevOut&, bool all_shadows);
cudaError_t launch_level(const DevScene&, const DevCamera&, const DevShade&, const DevWork&, const DevOut&, const DevWave&, int sms, cudaStream_t, DevCounters* shadow_counters);
cudaError_t launch_gather(const SpawnRec* recs, const uint32_t* nspec, double* rad_parent, const double* rad_child, uint64_t n_upper, cudaStream_t);
cudaError_t launch_resolve(const DevWork&, const DevOut&, cudaStream_t);
cudaError_t launch_export_li(const DevWork&, const DevOut&, const DevWave&, cudaStream_t);
cudaError_t launch_trace(const DevScene&, const TraceBox&, const double* rays, uint64_t n, uint32_t* ids, double* ts, double* ng, double* ns, cudaStream_t);
cudaError_t launch_l2_read(const void* buf, uint64_t bytes, int iters, float* sink, int sms, cudaStream_t);
cudaError_t launch_fp32_peak(int iters, float* sink, int sms, cudaStream_t);
cudaError_t launch_fp64_peak(int iters, double* sink, int sms, cudaStream_t);
cudaError_t launch_fastmath(const double* x, uint64_t n, double* rcp, double* rsq, cudaStream_t);
cudaError_t launch_flag_signal(void* flag, uint32_t value, cudaStream_t);
cudaError_t launch_flag_wait(const void* flags, uint32_t first, uint32_t n, uint32_t stride_bytes, uint32_t value, cudaStream_t);
}  // namespace lgb

using namespace lgb;

// The layouts the bindings mirror by hand (INTEGRATION.md, lasgun_b200/_native.py, tests/test_abi.py).
static_assert(sizeof(lgb_material) == 72 && offsetof(lgb_material, kind) == 64, "lgb_material layout (ABI v4)");
static_assert(sizeof(lgb_node) == 32 && sizeof(lgb_instance) == 16 + 2 * 16 * 8, "lgb_node / lgb_instance layout");
static_assert(sizeof(lgb_stats) == 21 * 8 + 12 * 4 + 8, "lgb_stats layout");
static_assert(sizeof(SpawnRec) == 72, "SpawnRec layout");
static_assert(sizeof(lgb_kernel_time) == 40 + 8 + 11 * 8, "lgb_kernel_time layout");

static thread_local std::string g_init_error;

struct DevBuf {
    void* p = nullptr; size_t cap = 0;
    cudaError_t reserve(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        cudaError_t e = cudaMalloc(&p, bytes);
        if (e == cudaSuccess) cap = bytes;
        return e;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

struct lgb_ctx {
    int device = 0;
    int sm_count = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev2 = nullptr;
    cudaEvent_t phase[kRenderEvents] = {};
    std::string error;
    DevBuf aov_li, beam2;
    DevBuf radiance, film, counters, tiles, aov_id, aov_t, aov_occl, scratch, wave, wave_ctr, ties, beam;
    DevBuf scene_copy;                     // the DevScene of the launches in flight, in global memory (DevScene::self, sync_scene_copy)
    // levels of the specular ray trees (Whitted recursion): radiance and spawn records of every level (kept until the fold back up),
    // the rays of the current and the next level, the wavefront buffers of the current level, per-level counters
    DevBuf lvl_rad[kMaxRecursion + 1], lvl_recs[kMaxRecursion + 1], raybuf[2], wave2, wave2_ctr, lvl_ctr;
    KernelLog klog{}; DevBuf klog_snaps;   // lgb_capture_profile
    // device group (lgb_init_devices): this context leads, `peers` render their share of the tiles into its film over NVLink
    std::vector<lgb_ctx*> peers;
    lgb_ctx* leader = nullptr;
    cudaMemPool_t share_pool = nullptr;    // a group leader's scene arenas and grids live here: a pool of its own that the peers may read (lgb_init_devices)
    std::mutex lazy_mu;                    // the caller's reference_tree callback is entered by one device at a time
    SideStreams side{};                    // streams the shadow chains of different lights are spread over (LGB_OPT_SIDE_STREAMS)
    int side_streams = 1;
    int whitted_wavefront = 1;             // LGB_OPT_WHITTED: 1 level-by-level wavefront, 0 one thread per ray tree (k_secondary)
    int beams = -1;                        // LGB_OPT_BEAMS: 0 off, 1 on, -1 automatic
    uint64_t wave_budget = 16ull << 30;    // LGB_OPT_WAVE_BUDGET_MB: bytes of per-sample buffers one band of a frame may take
    int setup_in_primary = 1;              // env LGB_SETUP_IN_PRIMARY (experiments): k_cprimary<SETUP>
    int lazy_bvh = -1;                     // LGB_OPT_LAZY_BVH: 0 build the device BVH at scene creation, 1 / -1 only when something needs it
    int camera_grid = -1;                  // LGB_OPT_CAMERA_GRID: 0 off, 1 on, -1 automatic
    int light_grids = -1;                  // LGB_OPT_LIGHT_GRIDS: 0 off, 1 on, -1 automatic (scenes of >= 1024 BVH nodes, <= 8 lights)
    std::vector<uint32_t> tile_host;
    uint32_t tile_key[4] = {0, 0, 0, 0};   // w, h, rank, ranks of the cached tile list
    uint32_t tile_count = 0;
    int count_work = 0;                    // LGB_OPT_COUNT_WORK
    void* staging = nullptr; size_t staging_cap = 0;   // pinned host buffer the scene arrays are assembled in
    cudaError_t reserve_staging(size_t bytes) {
        if (bytes <= staging_cap) return cudaSuccess;
        if (staging) cudaFreeHost(staging);
        staging = nullptr; staging_cap = 0;
        cudaError_t e = cudaHostAlloc(&staging, bytes + bytes / 4, cudaHostAllocDefault);
        if (e == cudaSuccess) staging_cap = bytes + bytes / 4;
        return e;
    }
    // pinned bounce buffer of the film read-back into pageable memory (finish_host), and one event per chunk of it
    void* film_host = nullptr; size_t film_host_cap = 0;
    std::vector<cudaEvent_t> chunk_ev;
    cudaStream_t copy_stream = nullptr;    // the film's slices travel here while the next slice is shaded (run_capture)
    bool host_film_done = false;           // run_capture delivered the film to CaptureArgs::host_film itself
    cudaError_t reserve_film_host(size_t bytes) {
        if (film_host_cap >= bytes) return cudaSuccess;
        if (film_host) cudaFreeHost(film_host);
        film_host = nullptr; film_host_cap = 0;
        cudaError_t e = cudaHostAlloc(&film_host, bytes, cudaHostAllocDefault);
        if (e == cudaSuccess) film_host_cap = bytes;
        return e;
    }
    cudaError_t reserve_chunk_events(size_t n) {
        while (chunk_ev.size() < n) { cudaEvent_t e; if (cudaError_t rc = cudaEventCreateWithFlags(&e, cudaEventDisableTiming)) return rc; chunk_ev.push_back(e); }
        return cudaSuccess;
    }
};

struct lgb_scene {
    lgb_ctx* ctx = nullptr;
    void* arena = nullptr;     // one stream-ordered device allocation holding every array of the scene
    bool owns_arena = true;    // false: imported (lgb_scene_import), the caller owns the memory
    bool gpu_built = false;    // the device BVH was built on the device (lgb_gpubuild.cu)
    // lazy reference tree (lasgun_b200.h): asked for only when a frame holds an exact-t tie
    lgb_reference_tree_fn lazy_fn = nullptr; void* lazy_user = nullptr;
    lgb_scene_desc lazy_desc{};                      // the caller's primitive / id arrays (they stay valid for the scene's lifetime)
    void* rank_buf = nullptr;                        // rank tables uploaded later live outside the arena
    uint64_t tie_retraces = 0;
    uint64_t bytes = 0;
    // camera grid (lgb_grid.cu) of the film size it was last built for; rebuilt when the film changes
    struct CamGrid { uint32_t w = 0, h = 0, shift = 0, nx = 0, n_large = 0; bool valid = false, refused = false; void* starts = nullptr; void* entries = nullptr; void* large = nullptr; uint64_t bytes = 0; double build_ms = 0; } camgrid;
    CamGrid& cam_grid() { return camgrid; }
    std::vector<void*> grid_allocs;    // light grids (lgb_grid.cu): table + per-light cell starts / entries / large lists, outside the arena
    struct GridHost { void* starts; void* entries; void* large; size_t starts_bytes, entries_bytes, large_bytes; uint32_t res, n_large; };
    std::vector<GridHost> grid_host;   // the same buffers with their sizes (device-group replication copies them to the peers)
    void* grid_table = nullptr;
    uint64_t expect_samples = 0;       // lgb_scene_desc.expected_film_pixels x spp (0: unknown, the scene may serve many frames)
    // deferred device BVH (LGB_OPT_LAZY_BVH): a plastic scene whose primary and shadow rays go through the grids never walks a tree, so
    // lgb_scene_create stores the primitives in the caller's order, keeps the uploaded raw arrays and the item boxes, and ensure_bvh
    // builds the tree (and re-orders the primitives, and rebuilds the grids) only if some entry point needs one
    struct Deferred { void* scratch = nullptr; RawScene raw{}; GItem* items = nullptr; GItem* final_items = nullptr; LeafArrays la{};
                      void* build_temp = nullptr; size_t build_bytes = 0, o_nodes = 0; uint32_t n = 0; double padd = 0; } deferred;
    double t_grids = 0;                // ms
    uint64_t grid_bytes = 0;
    std::vector<lgb_scene*> replicas;  // device group: the same scene on every peer, in peer order (arena copied over NVLink, not rebuilt)
    cudaEvent_t last_use = nullptr;   // recorded behind every capture on the stream it ran on: lgb_scene_destroy frees the arena behind it
    DevScene dev{};
    DevCamera cam{};
    DevShade shade{};
    double max_abs = 0.0;      // max |coordinate| over geometry, camera origin and lights
    // world box (scene and camera) the f32 error bound of every space was derived from: the traversal is conservative for rays
    // whose f32 origin lies inside it, so lgb_trace_rays starts the f32 ray of a caller-supplied origin outside where it enters it
    double origin_lo[3] = {0, 0, 0}, origin_hi[3] = {0, 0, 0};
    double build_ms = 0.0;     // host time of the device-BVH build inside lgb_scene_create
    double t_validate = 0, t_rank = 0, t_build = 0, t_convert_upload = 0, t_total = 0;   // ms, lgb_scene_create phases
};

static int fail(lgb_ctx* ctx, int code, const std::string& msg) {
    if (ctx) ctx->error = msg; else g_init_error = msg;
    return code;
}
static int cuda_fail(lgb_ctx* ctx, cudaError_t e, const char* what) {
    if (e == cudaErrorMemoryAllocation) { cudaGetLastError(); return fail(ctx, LGB_ERR_NOMEM, std::string(what) + ": out of device memory"); }
    return fail(ctx, LGB_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
}
#define CU(ctx, call) do { cudaError_t e__ = (call); if (e__ != cudaSuccess) return cuda_fail(ctx, e__, #call); } while (0)

extern "C" {

const char* lgb_status_string(int s) {
    switch (s) {
    case LGB_OK: return "ok";
    case LGB_ERR_INVALID: return "invalid argument";
    case LGB_ERR_CUDA: return "CUDA error";
    case LGB_ERR_UNSUPPORTED: return "unsupported on the device path";
    case LGB_ERR_NOMEM: return "out of memory";
    case LGB_ERR_NO_DEVICE: return "no sm_100 device";
    default: return "unknown status";
    }
}

int lgb_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

const char* lgb_last_error(lgb_ctx* ctx) { return ctx ? ctx->error.c_str() : g_init_error.c_str(); }

int lgb_init(int device, lgb_ctx** out) {
    if (!out) return fail(nullptr, LGB_ERR_INVALID, "lgb_init: out is NULL");
    *out = nullptr;
    int n = lgb_device_count();
    if (n <= 0) return fail(nullptr, LGB_ERR_NO_DEVICE, "lgb_init: no CUDA device visible (this library has no CPU fallback)");
    if (device < 0 || device >= n) return fail(nullptr, LGB_ERR_INVALID, "lgb_init: device index out of range");
    cudaDeviceProp prop;
    CU(nullptr, cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10) return fail(nullptr, LGB_ERR_NO_DEVICE, "lgb_init: device is not sm_100-class; kernels are built for sm_100a only");
    CU(nullptr, cudaSetDevice(device));
    lgb_ctx* c = new lgb_ctx();
    c->device = device;
    c->sm_count = prop.multiProcessorCount;
    if (const char* e = std::getenv("LGB_STACK_LIMIT")) {          // experiments: the per-thread local-memory size the driver lays the stacks out with
        size_t before = 0; cudaDeviceGetLimit(&before, cudaLimitStackSize);
        cudaDeviceSetLimit(cudaLimitStackSize, (size_t)std::atol(e));
        size_t after = 0; cudaDeviceGetLimit(&after, cudaLimitStackSize);
        std::fprintf(stderr, "[lgb_init] cudaLimitStackSize %zu -> %zu\n", before, after);
    }
    if (const char* e = std::getenv("LGB_BEAMS")) { const int v = std::atoi(e); c->beams = v < 0 ? -1 : (v != 0); }
    if (const char* e = std::getenv("LGB_LIGHT_GRIDS")) { const int v = std::atoi(e); c->light_grids = v < 0 ? -1 : (v != 0); }
    if (const char* e = std::getenv("LGB_WAVE_BUDGET_MB")) { const long v = std::atol(e); if (v >= 1) c->wave_budget = (uint64_t)v << 20; }
    if (const char* e = std::getenv("LGB_SETUP_IN_PRIMARY")) c->setup_in_primary = std::atoi(e) != 0;
    if (const char* e = std::getenv("LGB_LAZY_BVH")) { const int v = std::atoi(e); c->lazy_bvh = v < 0 ? -1 : (v != 0); }
    if (const char* e = std::getenv("LGB_CAMERA_GRID")) { const int v = std::atoi(e); c->camera_grid = v < 0 ? -1 : (v != 0); }
    c->side.n = 1;                         // one side stream: two lights' chains at a time (a third stream measured no further gain)
    cudaError_t ie = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
    if (ie == cudaSuccess) ie = cudaEventCreate(&c->ev0);
    if (ie == cudaSuccess) ie = cudaEventCreate(&c->ev1);
    if (ie == cudaSuccess) ie = cudaEventCreate(&c->ev2);
    for (auto& e : c->phase) if (ie == cudaSuccess) ie = cudaEventCreate(&e);
    for (int k = 0; k < c->side.n; k++) {
        if (ie == cudaSuccess) ie = cudaStreamCreateWithFlags(&c->side.s[k], cudaStreamNonBlocking);
        if (ie == cudaSuccess) ie = cudaEventCreateWithFlags(&c->side.join[k], cudaEventDisableTiming);
    }
    if (ie == cudaSuccess) ie = cudaEventCreateWithFlags(&c->side.fork, cudaEventDisableTiming);
    if (ie != cudaSuccess) {               // nothing of a half-made context survives (every handle below is NULL-safe to skip)
        if (c->stream) cudaStreamDestroy(c->stream);
        for (cudaEvent_t e : {c->ev0, c->ev1, c->ev2, c->side.fork}) if (e) cudaEventDestroy(e);
        for (auto& e : c->phase) if (e) cudaEventDestroy(e);
        for (int k = 0; k < c->side.n; k++) { if (c->side.s[k]) cudaStreamDestroy(c->side.s[k]); if (c->side.join[k]) cudaEventDestroy(c->side.join[k]); }
        delete c;
        return cuda_fail(nullptr, ie, "lgb_init: stream / event creation");
    }
    {   // scene arenas come from the stream-ordered pool and are kept cached between scenes (cudaMalloc/cudaFree cost ms)
        cudaMemPool_t mp;
        if (cudaDeviceGetDefaultMemPool(&mp, device) == cudaSuccess) {
            uint64_t keep = ~0ull;
            cudaMemPoolSetAttribute(mp, cudaMemPoolAttrReleaseThreshold, &keep);
        }
    }
    *out = c;
    return LGB_OK;
}

int lgb_init_devices(int ndev, const int* devices, lgb_ctx** out) {
    if (!out) return fail(nullptr, LGB_ERR_INVALID, "lgb_init_devices: out is NULL");
    *out = nullptr;
    if (ndev < 1 || !devices) return fail(nullptr, LGB_ERR_INVALID, "lgb_init_devices: empty device list");
    for (int i = 0; i < ndev; i++) for (int j = 0; j < i; j++) if (devices[i] == devices[j]) return fail(nullptr, LGB_ERR_INVALID, "lgb_init_devices: device listed twice");
    lgb_ctx* lead = nullptr;
    if (int rc = lgb_init(devices[0], &lead)) return rc;
    for (int i = 1; i < ndev; i++) {
        lgb_ctx* p = nullptr;
        int rc = lgb_init(devices[i], &p);
        if (!rc) {
            // the peer's kernels store their pixels into the leader's film: that needs direct peer access (NVLink / NVSwitch)
            int can = 0;
            cudaError_t e = cudaDeviceCanAccessPeer(&can, devices[i], devices[0]);
            if (e == cudaSuccess && can) {
                cudaSetDevice(devices[i]);
                e = cudaDeviceEnablePeerAccess(devices[0], 0);
                if (e == cudaErrorPeerAccessAlreadyEnabled) { cudaGetLastError(); e = cudaSuccess; }
            }
            if (e != cudaSuccess) rc = cuda_fail(nullptr, e, "lgb_init_devices: peer access");
            else if (!can) rc = fail(nullptr, LGB_ERR_UNSUPPORTED, "lgb_init_devices: a listed device cannot access the first one's memory (no NVLink / P2P path)");
        }
        if (rc) { const std::string msg = g_init_error; if (p) lgb_shutdown(p); lgb_shutdown(lead); g_init_error = msg; return rc; }
        p->leader = lead; p->beams = lead->beams; p->light_grids = lead->light_grids; p->camera_grid = lead->camera_grid; p->wave_budget = lead->wave_budget; p->lazy_bvh = lead->lazy_bvh; p->setup_in_primary = lead->setup_in_primary;
        lead->peers.push_back(p);
    }
    if (ndev > 1) {
        // What the peers copy from the leader (scene arena, light grids) is stream-ordered pool memory, which cudaDeviceEnablePeerAccess
        // does not cover: without a grant those peer copies are staged through the host (measured: 31 ms for 7 x 160 MB instead of ~2).
        // The grant goes to a pool of the group's own, made here while it is empty -- granting it on the device's default pool made
        // that pool refuse to grow afterwards whenever it already held memory of another context (scripts/diag_group_pool.py).
        cudaSetDevice(devices[0]);
        cudaMemPoolProps props{};
        props.allocType = cudaMemAllocationTypePinned; props.handleTypes = cudaMemHandleTypeNone;
        props.location.type = cudaMemLocationTypeDevice; props.location.id = devices[0];
        cudaError_t e = cudaMemPoolCreate(&lead->share_pool, &props);
        if (e == cudaSuccess) {
            uint64_t keep = ~0ull;
            cudaMemPoolSetAttribute(lead->share_pool, cudaMemPoolAttrReleaseThreshold, &keep);
            std::vector<cudaMemAccessDesc> acc((size_t)ndev - 1);
            for (int i = 1; i < ndev; i++) { acc[i - 1] = cudaMemAccessDesc{}; acc[i - 1].location.type = cudaMemLocationTypeDevice; acc[i - 1].location.id = devices[i]; acc[i - 1].flags = cudaMemAccessFlagsProtReadWrite; }
            e = cudaMemPoolSetAccess(lead->share_pool, acc.data(), acc.size());
        }
        if (e != cudaSuccess) { const int rc = cuda_fail(nullptr, e, "lgb_init_devices: shared memory pool"); const std::string msg = g_init_error; lgb_shutdown(lead); g_init_error = msg; return rc; }
    }
    *out = lead;
    return LGB_OK;
}
int lgb_context_devices(const lgb_ctx* c) { return c ? 1 + (int)c->peers.size() : 0; }

int lgb_film_alloc_shared(lgb_ctx* c, uint64_t bytes, void** d_film, uint8_t handle_out[LGB_IPC_HANDLE_BYTES]) {
    static_assert(sizeof(cudaIpcMemHandle_t) == LGB_IPC_HANDLE_BYTES, "IPC handle size");
    if (!c || !bytes || !d_film || !handle_out) return fail(c, LGB_ERR_INVALID, "lgb_film_alloc_shared: bad argument");
    CU(c, cudaSetDevice(c->device));
    void* p = nullptr;
    CU(c, cudaMalloc(&p, bytes));                       // IPC handles need a whole cudaMalloc allocation (no pool, no sub-allocation)
    cudaIpcMemHandle_t h;
    cudaError_t e = cudaIpcGetMemHandle(&h, p);
    if (e != cudaSuccess) { cudaFree(p); return cuda_fail(c, e, "cudaIpcGetMemHandle"); }
    std::memcpy(handle_out, &h, sizeof h);
    *d_film = p;
    return LGB_OK;
}
int lgb_film_open_shared(lgb_ctx* c, const uint8_t handle[LGB_IPC_HANDLE_BYTES], void** d_film) {
    if (!c || !handle || !d_film) return fail(c, LGB_ERR_INVALID, "lgb_film_open_shared: bad argument");
    CU(c, cudaSetDevice(c->device));
    cudaIpcMemHandle_t h; std::memcpy(&h, handle, sizeof h);
    CU(c, cudaIpcOpenMemHandle(d_film, h, cudaIpcMemLazyEnablePeerAccess));
    return LGB_OK;
}
int lgb_film_signal(lgb_ctx* c, void* d_flag, uint32_t value, void* stream) {
    if (!c || !d_flag) return fail(c, LGB_ERR_INVALID, "lgb_film_signal: NULL argument");
    CU(c, cudaSetDevice(c->device));
    CU(c, launch_flag_signal(d_flag, value, stream ? (cudaStream_t)stream : c->stream));
    return LGB_OK;
}
int lgb_film_wait(lgb_ctx* c, const void* d_flags, uint32_t first, uint32_t n, uint32_t stride_bytes, uint32_t value, void* stream) {
    if (!c || !d_flags || n > 1024 || stride_bytes % 4) return fail(c, LGB_ERR_INVALID, "lgb_film_wait: bad argument");
    CU(c, cudaSetDevice(c->device));
    CU(c, launch_flag_wait(d_flags, first, n, stride_bytes, value, stream ? (cudaStream_t)stream : c->stream));
    return LGB_OK;
}
int lgb_film_release_shared(lgb_ctx* c, void* d_film, int owner) {
    if (!c || !d_film) return LGB_ERR_INVALID;
    CU(c, cudaSetDevice(c->device));
    CU(c, cudaStreamSynchronize(c->stream));
    if (owner) CU(c, cudaFree(d_film)); else CU(c, cudaIpcCloseMemHandle(d_film));
    return LGB_OK;
}

int lgb_set_option(lgb_ctx* c, int option, int value) {
    if (!c) return LGB_ERR_INVALID;
    for (lgb_ctx* p : c->peers) lgb_set_option(p, option, value);
    if (option == LGB_OPT_COUNT_WORK) { c->count_work = value != 0; return LGB_OK; }
    if (option == LGB_OPT_BEAMS) { c->beams = value < 0 ? -1 : (value != 0); return LGB_OK; }
    if (option == LGB_OPT_WHITTED) { c->whitted_wavefront = value != 0; return LGB_OK; }
    if (option == LGB_OPT_SIDE_STREAMS) { c->side_streams = value != 0; return LGB_OK; }
    if (option == LGB_OPT_LIGHT_GRIDS) { c->light_grids = value < 0 ? -1 : (value != 0); return LGB_OK; }
    if (option == LGB_OPT_CAMERA_GRID) { c->camera_grid = value < 0 ? -1 : (value != 0); return LGB_OK; }
    if (option == LGB_OPT_LAZY_BVH) { c->lazy_bvh = value < 0 ? -1 : (value != 0); return LGB_OK; }
    if (option == LGB_OPT_WAVE_BUDGET_MB) { if (value < 1) return fail(c, LGB_ERR_INVALID, "lgb_set_option: budget must be at least 1 MB"); c->wave_budget = (uint64_t)value << 20; return LGB_OK; }
    return fail(c, LGB_ERR_INVALID, "lgb_set_option: unknown option");
}

void lgb_shutdown(lgb_ctx* c) {
    if (!c) return;
    for (lgb_ctx* p : c->peers) { p->leader = nullptr; lgb_shutdown(p); }
    c->peers.clear();
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    for (DevBuf* b : {&c->radiance, &c->film, &c->counters, &c->tiles, &c->aov_id, &c->aov_t, &c->aov_occl, &c->scratch, &c->wave, &c->wave_ctr, &c->ties, &c->beam, &c->raybuf[0], &c->raybuf[1], &c->wave2, &c->wave2_ctr, &c->lvl_ctr, &c->aov_li, &c->beam2, &c->scene_copy}) b->release();
    c->klog_snaps.release();
    for (int k = 0; k < c->klog.made; k++) { cudaEventDestroy(c->klog.ev0[k]); cudaEventDestroy(c->klog.ev1[k]); }
    for (DevBuf& b : c->lvl_rad) b.release();
    for (DevBuf& b : c->lvl_recs) b.release();
    if (c->staging) cudaFreeHost(c->staging);
    if (c->film_host) cudaFreeHost(c->film_host);
    for (cudaEvent_t e : c->chunk_ev) cudaEventDestroy(e);
    if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
    cudaEventDestroy(c->ev0); cudaEventDestroy(c->ev1); cudaEventDestroy(c->ev2);
    for (auto& e : c->phase) cudaEventDestroy(e);
    for (int k = 0; k < c->side.n; k++) { cudaStreamDestroy(c->side.s[k]); cudaEventDestroy(c->side.join[k]); }
    cudaEventDestroy(c->side.fork);
    if (c->share_pool) cudaMemPoolDestroy(c->share_pool);
    cudaStreamDestroy(c->stream);
    delete c;
}

}  // extern "C"

// ---------------------------------------------------------------------------------------- scene
static inline float f32_down(double v) { float f = (float)v; if ((double)f > v) f = nextafterf(f, -INFINITY); return f; }
static inline float f32_up(double v) { float f = (float)v; if ((double)f < v) f = nextafterf(f, INFINITY); return f; }

static void make_prim_boxes(const lgb_scene_desc* d, raw_vector<PrimBox>& prims) {
    const size_t ns = d->n_spheres, nc = d->n_cuboids, nt = d->n_triangles;
    prims.resize(ns + nc + nt);
    Pool& pool = Pool::get();
    pool.for_range(ns, 1 << 14, [&](size_t b0, size_t e0, size_t) {
        for (size_t i = b0; i < e0; i++) {
            const lgb_sphere& sp = d->spheres[i]; PrimBox& b = prims[i]; b.type = LGB_PRIM_SPHERE; b.index = (uint32_t)i;
            for (int k = 0; k < 3; k++) { double lo = sp.center[k] - sp.radius, hi = sp.center[k] + sp.radius; b.lo[k] = f32_down(std::min(lo, hi)); b.hi[k] = f32_up(std::max(lo, hi)); }
        }
    });
    for (size_t i = 0; i < nc; i++) {
        const lgb_cuboid& c = d->cuboids[i]; PrimBox& b = prims[ns + i]; b.type = LGB_PRIM_CUBOID; b.index = (uint32_t)i;
        for (int k = 0; k < 3; k++) { b.lo[k] = f32_down(std::min(c.min[k], c.max[k])); b.hi[k] = f32_up(std::max(c.min[k], c.max[k])); }
    }
    pool.for_range(nt, 1 << 14, [&](size_t b0, size_t e0, size_t) {
        for (size_t i = b0; i < e0; i++) {
            const lgb_triangle& t = d->triangles[i]; PrimBox& b = prims[ns + nc + i]; b.type = LGB_PRIM_TRIANGLE; b.index = (uint32_t)i;
            for (int k = 0; k < 3; k++) { b.lo[k] = std::min(t.p0[k], std::min(t.p1[k], t.p2[k])); b.hi[k] = std::max(t.p0[k], std::max(t.p1[k], t.p2[k])); }
        }
    });
}

// The caller's reference tree: indices in range, pre-order layout, and the traversal stack the reference itself would
// need (bvh.rs:469: 64 entries, it panics beyond).  Returns LGB_OK or an error code with `msg` set.
static int validate_reference_tree(const lgb_scene_desc* d, std::string& msg) {
    for (uint64_t i = 0; i < d->n_instances; i++)
        if (d->instances[i].root_node >= d->n_nodes) { msg = "instance: root_node out of range"; return LGB_ERR_INVALID; }
    const uint64_t nn = d->n_nodes;
    std::vector<uint32_t> need(nn, 0);
    for (uint64_t ii = nn; ii-- > 0;) {
        const lgb_node& n = d->nodes[ii];
        if (n.b & LGB_LEAF_FLAG) {
            uint64_t cnt = n.b & ~LGB_LEAF_FLAG, first = n.a;
            if (first + cnt > d->n_prim_refs) { msg = "node: leaf range outside prim_refs"; return LGB_ERR_INVALID; }
            uint32_t k = 0, worst = 0;
            for (uint64_t j = 0; j < cnt; j++) {
                uint32_t ref = d->prim_refs[first + j], type = ref >> 30, idx = ref & 0x3FFFFFFFu;
                uint64_t lim = type == LGB_PRIM_SPHERE ? d->n_spheres : type == LGB_PRIM_CUBOID ? d->n_cuboids : type == LGB_PRIM_TRIANGLE ? d->n_triangles : d->n_instances;
                if (idx >= lim) { msg = "prim_refs: index out of range"; return LGB_ERR_INVALID; }
                if (type == LGB_PRIM_INSTANCE) {
                    uint32_t root = d->instances[idx].root_node;
                    if (root <= ii) { msg = "instance: child BVH nodes must follow the referencing leaf"; return LGB_ERR_INVALID; }
                    k++;
                    worst = std::max(worst, need[root]);
                }
            }
            need[ii] = k ? (k - 1) + std::max(1u, worst) : 0;   // k roots pushed, popped one at a time
        } else {
            if (n.b > 2) { msg = "node: split axis out of range"; return LGB_ERR_INVALID; }
            if (ii + 1 >= nn || n.a <= ii + 1 || n.a >= nn) { msg = "node: child index out of range (pre-order expected)"; return LGB_ERR_INVALID; }
            need[ii] = 1 + std::max(need[ii + 1], need[n.a]);
        }
    }
    if (need[0] > (uint32_t)kStackDepth) { msg = "BVH needs more than 64 traversal stack entries (the reference would panic, bvh.rs:469)"; return LGB_ERR_UNSUPPORTED; }
    return LGB_OK;
}

// Lazy scenes: fetch the reference tree from the caller, build the rank tables and make them resident.
static int ensure_rank_tables(lgb_ctx* ctx, lgb_scene* s) {
    if (s->dev.rank || !s->lazy_fn) return LGB_OK;
    std::lock_guard<std::mutex> lock((ctx->leader ? ctx->leader : ctx)->lazy_mu);      // device group: one caller of the callback at a time
    lgb_reference_tree tree{};
    if (s->lazy_fn(s->lazy_user, &tree) != 0 || !tree.nodes || !tree.n_nodes) return fail(ctx, LGB_ERR_INVALID, "reference_tree callback failed");
    lgb_scene_desc d = s->lazy_desc;
    d.nodes = tree.nodes; d.n_nodes = tree.n_nodes; d.prim_refs = tree.prim_refs; d.n_prim_refs = tree.n_prim_refs;
    d.instances = tree.instances; d.n_instances = tree.n_instances;
    for (uint64_t i = 0; i < d.n_instances; i++)
        if (!d.instances[i].identity || d.instances[i].swap_backface) return fail(ctx, LGB_ERR_INVALID, "lazy reference tree: transformed instances need the tree at lgb_scene_create");
    std::string msg;
    if (int rc = validate_reference_tree(&d, msg)) return fail(ctx, rc, "reference tree: " + msg);
    const uint32_t P = s->dev.prim_count;
    const size_t bytes = (size_t)8 * (P + 1) * 4;
    cudaError_t e = ctx->reserve_staging(bytes);
    if (e != cudaSuccess) return cuda_fail(ctx, e, "cudaHostAlloc");
    BuiltScene one; one.spaces.emplace_back(); one.inst_space.assign(d.n_instances, kNoSpace);
    if (!build_rank_tables(&d, P, one, (uint32_t*)ctx->staging))
        return fail(ctx, LGB_ERR_INVALID, "reference tree: primitive ids must be a permutation of 0..n-1 and every primitive must be referenced by exactly one leaf");
    CU(ctx, cudaMallocAsync(&s->rank_buf, bytes, ctx->stream));
    CU(ctx, cudaMemcpyAsync(s->rank_buf, ctx->staging, bytes, cudaMemcpyHostToDevice, ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    s->dev.rank = (const uint32_t*)s->rank_buf; s->dev.rank_items = P + 1;
    return LGB_OK;
}

extern "C" { static int ensure_bvh(lgb_ctx* ctx, lgb_scene* s); }      // (defined inside the extern "C" block below)
// ---- export / import: the arena is position independent once DevScene's pointers are written as offsets
namespace {
struct SceneLayout { uint64_t magic, arena_bytes; DevScene dev; DevCamera cam; DevShade shade; double max_abs; double origin_lo[3], origin_hi[3]; };
constexpr uint64_t kLayoutMagic = 0x4C47423253434E34ull;       // "LGB2SCN4"
constexpr uint64_t kNullOffset = ~0ull;
template <class F> void for_each_pointer(DevScene& d, F f) {
    f((const void*&)d.nodes); f((const void*&)d.sph32); f((const void*&)d.sph64); f((const void*&)d.sph_mat); f((const void*&)d.sph_id);
    f((const void*&)d.cub32); f((const void*&)d.cub64); f((const void*&)d.cub_mat); f((const void*&)d.cub_id);
    f((const void*&)d.tri); f((const void*&)d.tri_nrm); f((const void*&)d.rank); f((const void*&)d.materials); f((const void*&)d.lights);
    f((const void*&)d.spaces); f((const void*&)d.inst_space); f((const void*&)d.sph_space); f((const void*&)d.cub_space); f((const void*&)d.tri_space);
}
}  // namespace

extern "C" {

int lgb_build_probe(const lgb_scene_desc* d, lgb_build_info* out) {
    if (!d || !out || !d->n_nodes) return LGB_ERR_INVALID;
    std::memset(out, 0, sizeof *out);
    const uint32_t prim_count = (uint32_t)(d->n_spheres + d->n_cuboids + d->n_triangles);
    const int threads = Pool::get().threads();
    BuiltScene bs; std::string berr;
    double wlo[3], whi[3];
    for (int k = 0; k < 3; k++) { wlo[k] = d->nodes[0].lo[k]; whi[k] = d->nodes[0].hi[k]; }
    if (build_scene(d, wlo, whi, bs, berr)) return LGB_ERR_INVALID;
    auto t0 = std::chrono::steady_clock::now();
    std::vector<uint32_t> rank((size_t)8 * (prim_count + bs.spaces.size()));
    out->ranks_ok = build_rank_tables(d, prim_count, bs, rank.data()) ? 1 : 0;
    out->rank_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    out->build_ms = bs.build_ms; out->prims = prim_count;
    if (bs.spaces.size() > 1) { out->nodes = (uint32_t)bs.nodes.size(); out->boxes_ok = 1; return LGB_OK; }   // structural check below: single space
    raw_vector<PrimBox> prims; make_prim_boxes(d, prims);
    BuiltBVH bvh;
    if (build_sah(prims.data(), prims.size(), 0.0f, threads, bvh)) return LGB_ERR_INVALID;
    out->nodes = (uint32_t)bvh.nodes.size(); out->max_depth = bvh.max_depth;
    // verify: every primitive in exactly one leaf, leaf boxes contain their primitives, child boxes nest
    std::vector<uint8_t> seen[3];
    for (int t = 0; t < 3; t++) seen[t].assign(bvh.order[t].size(), 0);
    std::vector<std::vector<const PrimBox*>> by_type(3);
    for (const PrimBox& p : prims) { if (by_type[p.type].size() <= p.index) by_type[p.type].resize(p.index + 1); by_type[p.type][p.index] = &p; }
    bool ok = true; double cost = 0.0;
    struct E { uint32_t node; float lo[3], hi[3]; };
    std::vector<E> st; E root; root.node = 0; for (int k = 0; k < 3; k++) { root.lo[k] = -INFINITY; root.hi[k] = INFINITY; } st.push_back(root);
    auto area = [](const float* lo, const float* hi) { float x = hi[0] - lo[0], y = hi[1] - lo[1], z = hi[2] - lo[2]; return (double)(x * y + x * z + y * z); };
    double root_area = 0.0;
    while (!st.empty()) {
        E e = st.back(); st.pop_back();
        const HostNode& n = bvh.nodes[e.node];
        for (int c = 0; c < 2; c++) {
            const float* lo = n.v + 6 * c; const float* hi = n.v + 6 * c + 3; const uint32_t w = c ? n.c1 : n.c0;
            if (c == 1 && n.c1 == n.c0) continue;     // tiny scene: both children are the same leaf
            for (int k = 0; k < 3; k++) if (lo[k] < e.lo[k] || hi[k] > e.hi[k]) ok = false;
            if (e.node == 0) root_area += area(lo, hi);
            if (w & kLeafBit) {
                const uint32_t type = (w >> 29) & 3u, cnt = ((w >> 24) & 31u) + 1u, first = w & kLeafFirstMask;
                out->leaves++; out->max_leaf = std::max(out->max_leaf, cnt); cost += area(lo, hi) * cnt;
                for (uint32_t i = 0; i < cnt; i++) {
                    if (first + i >= bvh.order[type].size()) { ok = false; continue; }
                    if (seen[type][first + i]++) ok = false;
                    const PrimBox* p = by_type[type][bvh.order[type][first + i]];
                    for (int k = 0; k < 3; k++) if (p->lo[k] < lo[k] || p->hi[k] > hi[k]) ok = false;
                }
            } else {
                cost += area(lo, hi) * 1.0;
                E ch; ch.node = w; std::memcpy(ch.lo, lo, 12); std::memcpy(ch.hi, hi, 12); st.push_back(ch);
            }
        }
    }
    for (int t = 0; t < 3; t++) for (uint8_t v : seen[t]) if (v != 1) ok = false;
    out->boxes_ok = ok ? 1 : 0;
    out->sah_cost = root_area > 0 ? cost / root_area : 0.0;
    return LGB_OK;
}

int lgb_scene_verify(lgb_ctx* ctx, const lgb_scene* s, lgb_build_info* out) {
    if (!ctx || !s || !out || s->ctx != ctx) return fail(ctx, LGB_ERR_INVALID, "lgb_scene_verify: bad argument");
    if (s->dev.instanced) return fail(ctx, LGB_ERR_UNSUPPORTED, "lgb_scene_verify: single-space scenes only");
    if (int rc = ensure_bvh(ctx, const_cast<lgb_scene*>(s))) return rc;
    std::memset(out, 0, sizeof *out);
    CU(ctx, cudaSetDevice(ctx->device));
    const DevScene& S = s->dev;
    const uint32_t P = S.prim_count;
    std::vector<HostNode> nodes(S.n_nodes);
    CU(ctx, cudaMemcpy(nodes.data(), S.nodes, (size_t)S.n_nodes * 64, cudaMemcpyDeviceToHost));
    // per type: how many primitives, their boxes (from the exact records) and canonical ids, in leaf order
    uint32_t cnt[3] = {0, 0, 0};
    for (const HostNode& n : nodes) for (int c = 0; c < 2; c++) {
        const uint32_t w = c ? n.c1 : n.c0;
        if (w & kLeafBit) { const uint32_t t = (w >> 29) & 3u; if (t < 3) cnt[t] = std::max(cnt[t], (w & kLeafFirstMask) + ((w >> 24) & 31u) + 1u); }
    }
    std::vector<double> s64((size_t)4 * cnt[0]), c64((size_t)6 * cnt[1]);
    std::vector<float4> tri((size_t)3 * cnt[2]);
    std::vector<uint32_t> sid(cnt[0]), cid(cnt[1]);
    if (cnt[0]) { CU(ctx, cudaMemcpy(s64.data(), S.sph64, s64.size() * 8, cudaMemcpyDeviceToHost)); CU(ctx, cudaMemcpy(sid.data(), S.sph_id, sid.size() * 4, cudaMemcpyDeviceToHost)); }
    if (cnt[1]) { CU(ctx, cudaMemcpy(c64.data(), S.cub64, c64.size() * 8, cudaMemcpyDeviceToHost)); CU(ctx, cudaMemcpy(cid.data(), S.cub_id, cid.size() * 4, cudaMemcpyDeviceToHost)); }
    if (cnt[2]) CU(ctx, cudaMemcpy(tri.data(), S.tri, tri.size() * 16, cudaMemcpyDeviceToHost));
    bool ok = cnt[0] + cnt[1] + cnt[2] == P;
    std::vector<uint8_t> seen_id(P, 0), seen_slot[3];
    for (int t = 0; t < 3; t++) seen_slot[t].assign(cnt[t], 0);
    auto prim_box = [&](uint32_t t, uint32_t i, double* lo, double* hi, uint32_t& id) {
        if (t == 0) { for (int k = 0; k < 3; k++) { const double a = s64[4 * (size_t)i + k] - s64[4 * (size_t)i + 3], b = s64[4 * (size_t)i + k] + s64[4 * (size_t)i + 3]; lo[k] = std::min(a, b); hi[k] = std::max(a, b); } id = sid[i]; }
        else if (t == 1) { for (int k = 0; k < 3; k++) { lo[k] = std::min(c64[6 * (size_t)i + k], c64[6 * (size_t)i + 3 + k]); hi[k] = std::max(c64[6 * (size_t)i + k], c64[6 * (size_t)i + 3 + k]); } id = cid[i]; }
        else {
            const float4 a = tri[3 * (size_t)i], b = tri[3 * (size_t)i + 1], c = tri[3 * (size_t)i + 2];
            const float x[3][3] = {{a.x, a.y, a.z}, {b.x, b.y, b.z}, {c.x, c.y, c.z}};
            for (int k = 0; k < 3; k++) { lo[k] = std::min(x[0][k], std::min(x[1][k], x[2][k])); hi[k] = std::max(x[0][k], std::max(x[1][k], x[2][k])); }
            std::memcpy(&id, &a.w, 4);
        }
    };
    struct E { uint32_t node, depth; float lo[3], hi[3]; };
    std::vector<E> st; E root{}; root.node = 0; root.depth = 0; for (int k = 0; k < 3; k++) { root.lo[k] = -INFINITY; root.hi[k] = INFINITY; } st.push_back(root);
    auto area = [](const float* lo, const float* hi) { float x = hi[0] - lo[0], y = hi[1] - lo[1], z = hi[2] - lo[2]; return (double)(x * y + x * z + y * z); };
    double cost = 0.0, root_area = 0.0; uint64_t visited = 0;
    while (!st.empty() && ok) {
        const E e = st.back(); st.pop_back();
        if (e.node >= S.n_nodes || ++visited > S.n_nodes) { ok = false; break; }
        const HostNode& n = nodes[e.node];
        for (int c = 0; c < 2; c++) {
            const float* lo = n.v + 6 * c; const float* hi = n.v + 6 * c + 3; const uint32_t w = c ? n.c1 : n.c0;
            for (int k = 0; k < 3; k++) if (!(lo[k] >= e.lo[k] && hi[k] <= e.hi[k])) ok = false;
            if (e.node == 0) root_area += area(lo, hi);
            if (w & kLeafBit) {
                const uint32_t t = (w >> 29) & 3u, k = ((w >> 24) & 31u) + 1u, first = w & kLeafFirstMask;
                out->leaves++; out->max_leaf = std::max(out->max_leaf, k); out->max_depth = std::max(out->max_depth, e.depth + 1);
                cost += area(lo, hi) * k;
                if (t > 2 || first + k > cnt[t]) { ok = false; continue; }
                for (uint32_t i = 0; i < k; i++) {
                    double plo[3], phi[3]; uint32_t id = 0;
                    prim_box(t, first + i, plo, phi, id);
                    if (seen_slot[t][first + i]++) ok = false;
                    if (id >= P || seen_id[id]++) ok = false;
                    for (int a = 0; a < 3; a++) if (!(plo[a] >= (double)lo[a] && phi[a] <= (double)hi[a])) ok = false;
                }
            } else {
                cost += area(lo, hi);
                E ch{}; ch.node = w; ch.depth = e.depth + 1; std::memcpy(ch.lo, lo, 12); std::memcpy(ch.hi, hi, 12); st.push_back(ch);
            }
        }
    }
    for (uint32_t i = 0; i < P && ok; i++) if (seen_id[i] != 1) ok = false;
    out->nodes = S.n_nodes; out->prims = P; out->boxes_ok = ok ? 1 : 0; out->ranks_ok = s->gpu_built ? 1 : 0;
    out->sah_cost = root_area > 0 ? cost / root_area : 0.0; out->build_ms = s->build_ms;
    return LGB_OK;
}

void lgb_scene_destroy(lgb_scene* s) {
    if (!s) return;
    for (lgb_scene* r : s->replicas) lgb_scene_destroy(r);
    s->replicas.clear();
    cudaSetDevice(s->ctx->device);
    if (s->last_use) {                 // a capture may still be running on a caller-supplied stream (lgb_capture_device is asynchronous)
        cudaStreamWaitEvent(s->ctx->stream, s->last_use, 0);
        cudaEventDestroy(s->last_use);
    }
    if (s->deferred.scratch) cudaFreeAsync(s->deferred.scratch, s->ctx->stream);
    for (void* g : s->grid_allocs) cudaFreeAsync(g, s->ctx->stream);
    for (void* g : {s->camgrid.starts, s->camgrid.entries, s->camgrid.large}) if (g) cudaFreeAsync(g, s->ctx->stream);
    if (s->rank_buf) cudaFreeAsync(s->rank_buf, s->ctx->stream);
    if (s->arena && s->owns_arena) cudaFreeAsync(s->arena, s->ctx->stream);      // stream-ordered: later work of this context is behind it
    else if (s->arena) cudaStreamSynchronize(s->ctx->stream);                    // borrowed arena: the caller may free it right after
    delete s;
}
uint64_t lgb_scene_device_bytes(const lgb_scene* s) { return s ? s->bytes + s->grid_bytes : 0; }

uint64_t lgb_scene_layout_bytes(void) { return sizeof(SceneLayout); }
int lgb_scene_export(const lgb_scene* s, void* layout_out, uint64_t layout_bytes, void** arena_dev, uint64_t* arena_bytes) {
    if (!s || !layout_out || layout_bytes < sizeof(SceneLayout) || !arena_dev || !arena_bytes) return LGB_ERR_INVALID;
    if (s->lazy_fn) return LGB_ERR_UNSUPPORTED;       // a lazy scene's rank tables live outside the arena: create it with the tree to replicate it
    if (int rc = ensure_bvh(s->ctx, const_cast<lgb_scene*>(s))) return rc;          // (an importer cannot build the tree: it has no item boxes)
    SceneLayout L{};
    L.magic = kLayoutMagic; L.arena_bytes = s->bytes; L.dev = s->dev; L.cam = s->cam; L.shade = s->shade; L.max_abs = s->max_abs;
    std::memcpy(L.origin_lo, s->origin_lo, sizeof L.origin_lo); std::memcpy(L.origin_hi, s->origin_hi, sizeof L.origin_hi);
    const char* base = (const char*)s->arena;
    L.dev.grids = nullptr;                             // light grids live outside the arena: the importer builds its own
    for_each_pointer(L.dev, [&](const void*& p) { p = (const void*)(p ? (uint64_t)((const char*)p - base) : kNullOffset); });
    std::memcpy(layout_out, &L, sizeof L);
    *arena_dev = s->arena; *arena_bytes = s->bytes;
    return LGB_OK;
}
static int build_light_grids(lgb_ctx* ctx, lgb_scene* s);
int lgb_scene_import(lgb_ctx* ctx, const void* layout, uint64_t layout_bytes, void* arena_dev, lgb_scene** out) {
    if (!ctx || !layout || layout_bytes < sizeof(SceneLayout) || !arena_dev || !out) return fail(ctx, LGB_ERR_INVALID, "lgb_scene_import: bad argument");
    SceneLayout L; std::memcpy(&L, layout, sizeof L);
    if (L.magic != kLayoutMagic) return fail(ctx, LGB_ERR_INVALID, "lgb_scene_import: not a scene layout of this library version");
    lgb_scene* s = new lgb_scene();
    s->ctx = ctx; s->arena = arena_dev; s->owns_arena = false; s->bytes = L.arena_bytes;
    s->dev = L.dev; s->cam = L.cam; s->shade = L.shade; s->max_abs = L.max_abs;
    std::memcpy(s->origin_lo, L.origin_lo, sizeof s->origin_lo); std::memcpy(s->origin_hi, L.origin_hi, sizeof s->origin_hi);
    const char* base = (const char*)arena_dev;
    bool ok = true;
    // every array must lie inside the arena with its whole extent (counts recomputed from the leaf words would need the nodes:
    // the per-type counts are bounded by prim_count, which is what the kernels can index)
    const DevScene& Ld = L.dev;
    const uint64_t P = Ld.prim_count, nsp = Ld.n_spaces;
    auto within = [&](const void* p, uint64_t bytes) {
        const uint64_t off = (uint64_t)p;
        if (off == kNullOffset) return true;
        return off <= L.arena_bytes && bytes <= L.arena_bytes - off;
    };
    ok = ok && Ld.nodes != (const float4*)kNullOffset && within(Ld.nodes, (uint64_t)Ld.n_nodes * 64) && within(Ld.rank, (uint64_t)8 * Ld.rank_items * 4);
    ok = ok && within(Ld.materials, 0) && within(Ld.lights, (uint64_t)Ld.n_lights * 72) && within(Ld.spaces, Ld.instanced ? nsp * sizeof(DevSpace) : 0);
    ok = ok && Ld.n_lights <= LGB_MAX_LIGHTS && Ld.rank_items >= P;
    for_each_pointer(s->dev, [&](const void*& p) {
        const uint64_t off = (uint64_t)p;
        if (off == kNullOffset) p = nullptr; else if (off > L.arena_bytes) ok = false; else p = base + off;
    });
    if (!ok) { delete s; return fail(ctx, LGB_ERR_INVALID, "lgb_scene_import: an array of the layout does not lie inside the arena"); }
    s->dev.grids = nullptr;
    if (int rc = build_light_grids(ctx, s)) { lgb_scene_destroy(s); return rc; }
    *out = s;
    return LGB_OK;
}
double lgb_scene_build_ms(const lgb_scene* s) { return s ? s->build_ms : 0.0; }
uint32_t lgb_scene_node_count(const lgb_scene* s) { if (!s) return 0; ensure_bvh(s->ctx, const_cast<lgb_scene*>(s)); return s->dev.n_nodes; }   // (builds a deferred tree)

// Light grids (lgb_grid.cu) of a resident single-space scene, on the scene's own device and the context's stream.  A scene the
// grids do not suit (transformed aggregates, a tiny BVH, many lights, many huge primitives) simply keeps dev.grids == NULL and its
// shadow rays traverse the BVH.
// "a BVH of >= 1024 nodes", also for a scene whose tree is deferred (leaves hold up to 4 primitives: ~n / 2 nodes)
static bool large_scene(const DevScene& S) { return S.nodes ? S.n_nodes >= 1024u : (S.n_sph + S.n_cub + S.n_tri) / 2 >= 1024u; }

// memory a device group's peers copy from (scene arena, grids): the leader's shared pool; any other context: the device's default pool
static cudaError_t shared_alloc(lgb_ctx* ctx, void** p, size_t bytes, cudaStream_t st) {
    return ctx->share_pool ? cudaMallocFromPoolAsync(p, bytes, ctx->share_pool, st) : cudaMallocAsync(p, bytes, st);
}
static int build_light_grids(lgb_ctx* ctx, lgb_scene* s) {
    DevScene& S = s->dev;
    S.grids = nullptr;
    for (void* g : s->grid_allocs) cudaFreeAsync(g, ctx->stream);      // (a rebuild after ensure_bvh re-ordered the primitives)
    s->grid_allocs.clear(); s->grid_host.clear(); s->grid_table = nullptr; s->grid_bytes = 0;
    bool want = ctx->light_grids == 1 || (ctx->light_grids < 0 && large_scene(S) && S.n_lights <= 8u);
    // a scene made for ONE frame of known size (capture(scene, film)) must earn its grids within that frame: they cost about as much to
    // build as 10 shadow rays per primitive cost to trace (measured: `mesh1m`, 0.7 shadow rays per triangle, 3.8 ms of grids for 0.1 ms of render)
    if (want && ctx->light_grids < 0 && s->expect_samples && s->expect_samples * S.n_lights < 8ull * (S.n_sph + S.n_cub + S.n_tri)) want = false;
    if (!want || S.instanced || S.n_lights == 0 || S.n_sph + S.n_cub + S.n_tri == 0) return LGB_OK;
    auto t0 = std::chrono::steady_clock::now();
    CU(ctx, cudaSetDevice(ctx->device));
    uint32_t res = 1024;
    if (const char* e = std::getenv("LGB_GRID_RES")) res = std::min(4096u, std::max(16u, (uint32_t)std::atoi(e)));
    const uint32_t nl = S.n_lights;
    const size_t nc = grid_cells(res), scan_bytes = grid_scan_bytes(res);
    cudaStream_t st = ctx->stream;
    std::vector<void*> temp, mine;               // freed at the end | kept by the scene
    auto cleanup = [&](bool keep) {
        for (void* p : temp) cudaFreeAsync(p, st);
        if (!keep) for (void* p : mine) cudaFreeAsync(p, st);
    };
#define GR(call) do { cudaError_t e__ = (call); if (e__ != cudaSuccess) { cleanup(false); return cuda_fail(ctx, e__, #call); } } while (0)
    auto alloc = [&](std::vector<void*>& owner, size_t bytes, void** out) {
        cudaError_t e = &owner == &mine ? shared_alloc(ctx, out, std::max<size_t>(bytes, 16), st) : cudaMallocAsync(out, std::max<size_t>(bytes, 16), st);
        if (e == cudaSuccess) owner.push_back(*out);
        return e;
    };
    // Four allocations per scene, not twenty: the stream-ordered pool of a long-lived process is fragmented, and the per-light buffers
    // of `spheres1m` cost 5 ms to allocate as the bench's fourth workload against 1 ms in a fresh process.  One temporary block for the
    // count passes, one kept block for the table and every light's cell starts; after the totals are known one kept block for every
    // light's entries and large list, and one temporary block that the lights' fill + sort passes use in turn (same stream).
    auto up = [](size_t v) { return (v + 255) & ~(size_t)255; };
    const size_t b_counts = up((nc + 1) * 4), b_scan = up(scan_bytes), b_bounds = up(64 * 8 * (size_t)nl), b_totals = up(8 * (size_t)nl), b_large = up(sizeof(uint2) * kGridLargeCap * (size_t)nl);
    char* tmp_a = nullptr; char* keep_a = nullptr;
    GR(alloc(temp, b_counts + b_scan + b_bounds + b_totals + b_large, (void**)&tmp_a));
    uint32_t* counts = (uint32_t*)tmp_a; void* scan_tmp = tmp_a + b_counts; unsigned long long* bounds = (unsigned long long*)(tmp_a + b_counts + b_scan);
    uint32_t* totals = (uint32_t*)(tmp_a + b_counts + b_scan + b_bounds); uint2* large_tmp = (uint2*)(tmp_a + b_counts + b_scan + b_bounds + b_totals);
    const size_t b_tab = up(sizeof(DevGrid) * (size_t)nl), b_starts = up((nc + 1) * 4);
    GR(alloc(mine, b_tab + b_starts * nl, (void**)&keep_a));
    DevGrid* dtab = (DevGrid*)keep_a;
    GR(cudaMemsetAsync(dtab, 0, sizeof(DevGrid) * (size_t)nl, st));
    const bool timing = getenv("LGB_TIMING") != nullptr;
    auto lap = [&](const char* what) { if (!timing) return; cudaStreamSynchronize(st); fprintf(stderr, "[light grids]   %-28s %.2f ms\n", what, std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count()); };
    lap("temporaries allocated");
    std::vector<uint32_t*> starts(nl, nullptr);
    for (uint32_t l = 0; l < nl; l++) {          // face mappings, counts, scans of every light, then ONE synchronisation for the totals
        starts[l] = (uint32_t*)(keep_a + b_tab + b_starts * l);
        GR(grid_count(S, l, res, dtab + l, bounds + 64 * (size_t)l, counts, starts[l], scan_tmp, scan_bytes, large_tmp + (size_t)kGridLargeCap * l, totals + 2 * (size_t)l, st));
    }
    lap("bounds + counts + scans");
    std::vector<uint32_t> h_tot(2 * (size_t)nl);
    GR(cudaMemcpyAsync(h_tot.data(), totals, 8 * (size_t)nl, cudaMemcpyDeviceToHost, st));
    GR(cudaStreamSynchronize(st));
    bool ok = true;
    s->grid_host.clear();
    for (uint32_t l = 0; l < nl; l++) ok = ok && h_tot[2 * l + 1] <= kGridLargeCap;
    uint64_t bytes = 0, entries_all = 0;
    if (ok) {
        struct Head { const uint32_t* cell_start; const uint2* entries; const uint2* large; uint32_t res, n_large; };
        static_assert(offsetof(DevGrid, map) == sizeof(Head), "DevGrid head");
        std::vector<Head> heads(nl);
        size_t keep_b_bytes = 0, max_entries = 0, max_sort = 0;
        for (uint32_t l = 0; l < nl; l++) {
            const uint32_t total = h_tot[2 * l], n_large = h_tot[2 * l + 1];
            keep_b_bytes += up(std::max<size_t>(sizeof(uint2) * (size_t)total, 16)) + up(std::max<size_t>(sizeof(uint2) * (size_t)n_large, 16));
            max_entries = std::max(max_entries, up(std::max<size_t>(sizeof(uint2) * (size_t)total, 16)));
            max_sort = std::max(max_sort, up(grid_sort_bytes(total, nc)));
        }
        char* keep_b = nullptr; char* tmp_b = nullptr;
        GR(alloc(mine, keep_b_bytes, (void**)&keep_b));
        GR(alloc(temp, max_entries + max_sort, (void**)&tmp_b));
        size_t at = 0;
        for (uint32_t l = 0; l < nl; l++) {
            const uint32_t total = h_tot[2 * l], n_large = h_tot[2 * l + 1];
            uint2* entries = (uint2*)(keep_b + at); at += up(std::max<size_t>(sizeof(uint2) * (size_t)total, 16));
            uint2* large = (uint2*)(keep_b + at); at += up(std::max<size_t>(sizeof(uint2) * (size_t)n_large, 16));
            uint2* entries_tmp = (uint2*)tmp_b; void* sort_tmp = tmp_b + max_entries;
            const size_t sort_bytes = grid_sort_bytes(total, nc);
            GR(grid_fill(S, l, res, dtab + l, counts, starts[l], entries_tmp, entries, total, sort_tmp, sort_bytes, large_tmp + (size_t)kGridLargeCap * l, n_large, st));
            if (n_large) GR(cudaMemcpyAsync(large, large_tmp + (size_t)kGridLargeCap * l, sizeof(uint2) * n_large, cudaMemcpyDeviceToDevice, st));
            heads[l] = Head{starts[l], entries, large, res, n_large};
            s->grid_host.push_back(lgb_scene::GridHost{starts[l], entries, large, (nc + 1) * 4, sizeof(uint2) * (size_t)total, sizeof(uint2) * (size_t)n_large, res, n_large});
            bytes += (nc + 1) * 4 + sizeof(uint2) * ((size_t)total + n_large); entries_all += total;
        }
        lap("entries allocated, filled, sorted");
        for (uint32_t l = 0; l < nl; l++) GR(cudaMemcpyAsync((char*)(dtab + l), &heads[l], sizeof(Head), cudaMemcpyHostToDevice, st));
        GR(cudaStreamSynchronize(st));           // `heads` is on this stack frame; captures may run on other streams
        S.grids = dtab;
        s->grid_table = dtab;
        s->grid_allocs = mine;
        s->grid_bytes = bytes + sizeof(DevGrid) * nl;
    }
    cleanup(ok);
#undef GR
    s->t_grids = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    if (getenv("LGB_TIMING")) fprintf(stderr, "[light grids] %u lights, res %u, %llu entries, %.1f MB, %.2f ms (host clock, two synchronisations)%s\n", nl, res,
                                      (unsigned long long)entries_all, s->grid_bytes / 1e6, s->t_grids, ok ? "" : " REFUSED");
    return LGB_OK;
}

static int replicate_to_peers(lgb_ctx* ctx, lgb_scene* s);
// The device BVH of a scene created without one (lgb_scene::Deferred): binned-SAH build from the kept item boxes, the primitives
// re-written in leaf order, the grids (which index the primitive arrays) rebuilt, the peers of a device group re-supplied.
static int ensure_bvh(lgb_ctx* ctx, lgb_scene* s) {
    if (s->dev.nodes || !s->deferred.scratch) return LGB_OK;
    if (ctx->leader) return fail(ctx, LGB_ERR_INVALID, "internal: a device-group replica cannot build its own BVH (the leader re-supplies it)");
    auto t0 = std::chrono::steady_clock::now();
    CU(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    if (s->last_use) CU(ctx, cudaStreamWaitEvent(st, s->last_use, 0));       // a capture on a caller's stream may still read the arrays
    lgb_scene::Deferred& F = s->deferred;
    char* D = (char*)s->arena;
    GpuBuildInfo info{};
    uint32_t* typepos[3] = {nullptr, nullptr, nullptr};
    cudaError_t e = gpu_build_sah(F.items, F.n, (HostNode*)(D + F.o_nodes), F.final_items, typepos, F.build_temp, F.build_bytes, st, &info);
    if (e != cudaSuccess) return cuda_fail(ctx, e, "gpu_build_sah");
    if (info.max_depth + 1 > (uint32_t)kStackDepth) return fail(ctx, LGB_ERR_UNSUPPORTED, "device BVH deeper than the 64-entry traversal stack");
    if ((e = launch_convert(F.raw, F.la, F.final_items, F.n, typepos, F.padd, st)) != cudaSuccess) return cuda_fail(ctx, e, "k_convert");
    CU(ctx, cudaStreamSynchronize(st));
    cudaFreeAsync(F.scratch, st);
    F = lgb_scene::Deferred{};
    s->dev.nodes = (const float4*)(D + s->bytes); s->dev.n_nodes = info.n_nodes;      // (bytes == o_nodes while the tree was deferred)
    s->bytes += (size_t)info.n_nodes * 64;
    for (void** q : {&s->camgrid.starts, &s->camgrid.entries, &s->camgrid.large}) if (*q) { cudaFreeAsync(*q, st); *q = nullptr; }
    s->camgrid.valid = false; s->camgrid.refused = false;
    if (!ctx->peers.empty()) {
        for (lgb_scene* r : s->replicas) lgb_scene_destroy(r);
        s->replicas.clear();
        if (int rc = replicate_to_peers(ctx, s)) return rc;                 // (builds the leader's grids too)
    } else if (int rc = build_light_grids(ctx, s)) return rc;
    s->build_ms += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    if (getenv("LGB_TIMING")) fprintf(stderr, "[ensure_bvh] deferred device BVH built on demand: %u nodes, %.2f ms\n", info.n_nodes, std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count());
    return LGB_OK;
}

// Device group: the finished arena is copied to every peer over NVLink (one 61 MB peer copy each for `mixed4k`, not a rebuild) and
// the peer's scene points into its own copy.  A lazy scene stays lazy on every device (same callback, entered under one mutex).
static int replicate_to_peers(lgb_ctx* ctx, lgb_scene* s) {
    const char* base = (const char*)s->arena;
    for (lgb_ctx* p : ctx->peers) {
        CU(ctx, cudaSetDevice(p->device));
        void* arena = nullptr;
        CU(ctx, cudaMallocAsync(&arena, s->bytes, p->stream));
        lgb_scene* r = new lgb_scene();
        r->ctx = p; r->arena = arena; r->owns_arena = true; r->bytes = s->bytes; r->gpu_built = s->gpu_built;
        r->dev = s->dev; r->cam = s->cam; r->shade = s->shade; r->max_abs = s->max_abs;
        std::memcpy(r->origin_lo, s->origin_lo, sizeof r->origin_lo); std::memcpy(r->origin_hi, s->origin_hi, sizeof r->origin_hi);
        r->lazy_fn = s->lazy_fn; r->lazy_user = s->lazy_user; r->lazy_desc = s->lazy_desc;
        for_each_pointer(r->dev, [&](const void*& q) { if (q) q = (const char*)arena + ((const char*)q - base); });
        s->replicas.push_back(r);
        CU(ctx, cudaMemcpyPeerAsync(arena, p->device, s->arena, ctx->device, s->bytes, p->stream));
    }
    // the leader builds its light grids while the arenas travel; the grids then travel too (a table and three buffers per light:
    // 98 MB for `mixed4k`) and only the pointers of the peer's table are rewritten -- rebuilding them per device cost 12 ms at 8 GPUs
    if (int rc0 = build_light_grids(ctx, s)) return rc0;
    struct Head { const uint32_t* cell_start; const uint2* entries; const uint2* large; uint32_t res, n_large; };
    std::vector<std::vector<Head>> all_heads(ctx->peers.size());      // (alive until every peer's stream is drained below)
    for (size_t k = 0; k < ctx->peers.size(); k++) {
        lgb_ctx* p = ctx->peers[k];
        lgb_scene* r = s->replicas[k];
        r->dev.grids = nullptr;
        if (!s->dev.grids) continue;
        CU(ctx, cudaSetDevice(p->device));
        const size_t nl = s->grid_host.size();
        void* tab = nullptr;
        CU(ctx, cudaMallocAsync(&tab, sizeof(DevGrid) * nl, p->stream));
        r->grid_allocs.push_back(tab);
        CU(ctx, cudaMemcpyPeerAsync(tab, p->device, s->grid_table, ctx->device, sizeof(DevGrid) * nl, p->stream));
        std::vector<Head>& heads = all_heads[k];
        heads.resize(nl);
        for (size_t l = 0; l < nl; l++) {
            const lgb_scene::GridHost& g = s->grid_host[l];
            void* b[3] = {nullptr, nullptr, nullptr};
            const void* src[3] = {g.starts, g.entries, g.large};
            const size_t bytes[3] = {g.starts_bytes, g.entries_bytes, g.large_bytes};
            for (int q = 0; q < 3; q++) {
                CU(ctx, cudaMallocAsync(&b[q], std::max<size_t>(bytes[q], 16), p->stream));
                r->grid_allocs.push_back(b[q]);
                if (bytes[q]) CU(ctx, cudaMemcpyPeerAsync(b[q], p->device, src[q], ctx->device, bytes[q], p->stream));
            }
            heads[l] = Head{(const uint32_t*)b[0], (const uint2*)b[1], (const uint2*)b[2], g.res, g.n_large};
            r->grid_host.push_back(lgb_scene::GridHost{b[0], b[1], b[2], bytes[0], bytes[1], bytes[2], g.res, g.n_large});
        }
        for (size_t l = 0; l < nl; l++) CU(ctx, cudaMemcpyAsync((char*)tab + sizeof(DevGrid) * l, &heads[l], sizeof(Head), cudaMemcpyHostToDevice, p->stream));
        r->dev.grids = (const DevGrid*)tab; r->grid_table = tab; r->grid_bytes = s->grid_bytes;
    }
    for (lgb_ctx* p : ctx->peers) { CU(ctx, cudaSetDevice(p->device)); CU(ctx, cudaStreamSynchronize(p->stream)); }
    CU(ctx, cudaSetDevice(ctx->device));
    return LGB_OK;
}

int lgb_scene_create(lgb_ctx* ctx, const lgb_scene_desc* d, lgb_scene** out) {
    if (!ctx || !d || !out) return fail(ctx, LGB_ERR_INVALID, "lgb_scene_create: NULL argument");
    *out = nullptr;
    if (d->abi_version != LGB_ABI_VERSION) return fail(ctx, LGB_ERR_INVALID, "lgb_scene_create: abi_version mismatch");
    if (!d->reference_tree && (d->n_nodes == 0 || !d->nodes)) return fail(ctx, LGB_ERR_INVALID, "lgb_scene_create: empty BVH (the reference does not terminate on an empty aggregate, bvh.rs:240)");
    if (d->n_nodes >= (1ull << 31) || d->n_prim_refs >= (1ull << 32) || d->n_spheres >= (1ull << 30) || d->n_cuboids >= (1ull << 30) ||
        d->n_triangles >= (1ull << 30) || d->n_instances >= (1ull << 30))
        return fail(ctx, LGB_ERR_INVALID, "lgb_scene_create: array too large for 30-bit primitive references");
    if (d->n_lights > LGB_MAX_LIGHTS) return fail(ctx, LGB_ERR_UNSUPPORTED, "lgb_scene_create: more than LGB_MAX_LIGHTS point lights");
    if (d->n_materials == 0 && (d->n_spheres || d->n_cuboids || d->n_triangles)) return fail(ctx, LGB_ERR_INVALID, "lgb_scene_create: no materials");
    if (d->camera.supersampling_root == 0 || d->camera.supersampling_root > 256) return fail(ctx, LGB_ERR_INVALID, "lgb_scene_create: supersampling_root out of range");
    CU(ctx, cudaSetDevice(ctx->device));

    auto tc0 = std::chrono::steady_clock::now();
    auto ms_since = [](std::chrono::steady_clock::time_point t) { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t).count(); };
    // ---- materials: the device record (lgb_types.cuh) of every `Material::scattering` (material/*.rs)
    std::vector<double> mats(kMatStride * d->n_materials);
    bool any_general = false, any_specular = false;
    for (uint64_t i = 0; i < d->n_materials; i++) {
        const lgb_material& m = d->materials[i];
        if (m.kind > LGB_MAT_MIRROR) return fail(ctx, LGB_ERR_INVALID, "material: unknown kind");
        const bool plain = m.kind == LGB_MAT_PLASTIC || (m.kind == LGB_MAT_MATTE && m.roughness == 0.0);     // the lobes of the fast path
        const bool specular = m.kind == LGB_MAT_GLASS || m.kind == LGB_MAT_MIRROR;
        bool diffuse = m.kind == LGB_MAT_MATTE ? true : !(m.kd[0] == 0.0 && m.kd[1] == 0.0 && m.kd[2] == 0.0);   // plastic.rs:24, matte.rs:18-26
        bool glossy = m.kind == LGB_MAT_PLASTIC && !(m.ks[0] == 0.0 && m.ks[1] == 0.0 && m.ks[2] == 0.0);        // plastic.rs:29
        if (!plain) { diffuse = glossy = false; any_general = true; }
        any_specular |= specular;
        double* o = &mats[kMatStride * i];
        o[0] = m.kd[0]; o[1] = m.kd[1]; o[2] = m.kd[2]; o[3] = m.roughness;
        o[4] = m.ks[0]; o[5] = m.ks[1]; o[6] = m.ks[2];
        long long fl = (diffuse ? kMatDiffuse : 0) | (glossy ? kMatGlossy : 0) | (plain ? 0 : kMatGeneral) | (specular ? kMatSpecular : 0) | ((long long)m.kind << 8);
        std::memcpy(&o[7], &fl, 8);
        o[8] = m.roughness_v; o[9] = 0.0; o[10] = o[11] = 0.0;
        if (m.kind == LGB_MAT_MATTE && m.roughness != 0.0) {               // OrenNayar::new, diffuse.rs:28-34 (cgmath Deg -> Rad: deg * pi / 180)
            const double sigma = m.roughness * 3.14159265358979323846264338327950288 / 180.0;
            const double sigma2 = sigma * sigma;
            o[8] = 1.0 - (sigma2 / 2.0 * (sigma2 + 0.33));
            o[9] = 0.45 * sigma2 / (sigma2 + 0.09);
        }
    }
    if (any_specular && d->recursion > kMaxRecursion) return fail(ctx, LGB_ERR_UNSUPPORTED, "lgb_scene_create: recursion deeper than 12 with glass or mirror materials");
    auto mat_ok = [&](const uint32_t* arr, uint64_t n) { for (uint64_t i = 0; i < n; i++) if (arr[i] >= d->n_materials) return false; return true; };
    if ((d->n_spheres && (!d->spheres || !d->sphere_material || !d->sphere_id)) || (d->n_cuboids && (!d->cuboids || !d->cuboid_material || !d->cuboid_id)) ||
        (d->n_triangles && (!d->triangles || !d->triangle_material || !d->triangle_id)) || (d->n_instances && !d->instances) ||
        (d->n_prim_refs && !d->prim_refs) || (d->n_lights && !d->lights))
        return fail(ctx, LGB_ERR_INVALID, "lgb_scene_create: NULL array with non-zero count");
    if (!mat_ok(d->sphere_material, d->n_spheres) || !mat_ok(d->cuboid_material, d->n_cuboids) || !mat_ok(d->triangle_material, d->n_triangles))
        return fail(ctx, LGB_ERR_INVALID, "lgb_scene_create: material index out of range");

    // ---- the reference tree: given now, or on demand (lazy: only an exact-t tie ever needs it)
    lgb_scene_desc eager;                                    // lazy desc of a scene the device-side builder does not take: fetch the tree now
    const uint32_t prim_total = (uint32_t)(d->n_spheres + d->n_cuboids + d->n_triangles);
    bool lazy = !d->nodes && d->reference_tree;
    // (rays below specular hits break exact-t ties through resident rank tables: no lazy tree for scenes with glass or mirrors)
    if (lazy && (any_specular || !(prim_total >= 32768u && prim_total <= kLeafFirstMask && !std::getenv("LGB_HOST_BUILD")))) {
        lgb_reference_tree tree{};
        if (d->reference_tree(d->reference_tree_user, &tree) != 0 || !tree.nodes || !tree.n_nodes) return fail(ctx, LGB_ERR_INVALID, "lgb_scene_create: reference_tree callback failed");
        eager = *d;
        eager.nodes = tree.nodes; eager.n_nodes = tree.n_nodes; eager.prim_refs = tree.prim_refs; eager.n_prim_refs = tree.n_prim_refs;
        eager.instances = tree.instances; eager.n_instances = tree.n_instances;
        d = &eager; lazy = false;
    }
    if (!lazy) {
        if (d->n_nodes == 0 || !d->nodes) return fail(ctx, LGB_ERR_INVALID, "lgb_scene_create: empty BVH (the reference does not terminate on an empty aggregate, bvh.rs:240)");
        std::string vmsg;
        if (int vrc = validate_reference_tree(d, vmsg)) return fail(ctx, vrc, vmsg);
    } else if (!d->root.identity || d->root.swap_backface) return fail(ctx, LGB_ERR_INVALID, "lgb_scene_create: a lazy reference tree needs an untransformed root");

    lgb_scene* s = new lgb_scene();
    s->ctx = ctx;
    s->expect_samples = (uint64_t)d->expected_film_pixels * d->camera.supersampling_root * d->camera.supersampling_root;
    auto bail = [&](int code) { lgb_scene_destroy(s); return code; };

    // ---- box that contains the scene and every ray origin, in world coordinates: it bounds the coordinates an f32
    //      ray can carry in every space, hence the error bound of the conservative filters
    double wlo[3], whi[3];
    {
        double rlo[3], rhi[3];
        for (int k = 0; k < 3; k++) { rlo[k] = lazy ? d->bounds_lo[k] : (double)d->nodes[0].lo[k]; rhi[k] = lazy ? d->bounds_hi[k] : (double)d->nodes[0].hi[k]; }
        for (int k = 0; k < 3; k++) if (!(rlo[k] <= rhi[k]) || !std::isfinite(rlo[k]) || !std::isfinite(rhi[k])) return bail(fail(ctx, LGB_ERR_INVALID, "lgb_scene_create: bad scene bounds"));
        if (!d->root.identity) {                           // the root level's box is in the root aggregate's coordinates
            for (int r = 0; r < 3; r++) {
                double l = d->root.m[12 + r], h = l;
                for (int c = 0; c < 3; c++) { const double a = d->root.m[4 * c + r] * rlo[c], b = d->root.m[4 * c + r] * rhi[c]; l += std::min(a, b); h += std::max(a, b); }
                wlo[r] = l; whi[r] = h;
            }
        } else for (int k = 0; k < 3; k++) { wlo[k] = rlo[k]; whi[k] = rhi[k]; }
        // orthographic origins move across the image plane (camera.rs:126-128); aspect <= 4 assumed, checked per capture
        const double slack = 2.5 * std::fabs(d->camera.image_plane_height) * std::fabs(d->camera.pixel_separation);
        for (int k = 0; k < 3; k++) {
            if (std::isfinite(d->camera.origin[k])) { wlo[k] = std::min(wlo[k], d->camera.origin[k] - slack); whi[k] = std::max(whi[k], d->camera.origin[k] + slack); }
        }
        for (int k = 0; k < 3; k++) { s->origin_lo[k] = wlo[k]; s->origin_hi[k] = whi[k]; }
    }

    // ---- device acceleration structure: one binned-SAH BVH per space over the same primitives, rank tables from
    //      the caller's reference tree (lgb_build.hpp); everything is stored in leaf order.
    const uint32_t prim_count = (uint32_t)(d->n_spheres + d->n_cuboids + d->n_triangles);
    if (prim_count == 0) return bail(fail(ctx, LGB_ERR_INVALID, "lgb_scene_create: no primitives"));
    const int threads = Pool::get().threads();
    s->t_validate = ms_since(tc0);
    bool has_spaces = !d->root.identity || d->root.swap_backface;
    for (uint64_t i = 0; i < d->n_instances && !has_spaces; i++) has_spaces = !d->instances[i].identity || d->instances[i].swap_backface;
    // Large single-space scenes: the device BVH is built ON the device (lgb_gpubuild.cu); the host builder stays for
    // scenes with nested spaces and for small ones (LGB_HOST_BUILD=1 forces it: A/B runs and tests).
    const bool gpu_build = !has_spaces && prim_count >= 32768u && prim_count <= kLeafFirstMask && !std::getenv("LGB_HOST_BUILD");
    if (gpu_build) {
        auto tg0 = std::chrono::steady_clock::now();
        static_assert(sizeof(HostNode) == 64, "node layout");
        const size_t ns = d->n_spheres, ncb = d->n_cuboids, nt = d->n_triangles, n = prim_count;
        const bool any_normals = nt && d->tri_normals;
        double M = 0.0;
        auto upd = [&](double v) { const double a = std::fabs(v); if (a > M && std::isfinite(a)) M = a; };
        for (int k = 0; k < 3; k++) { upd(wlo[k]); upd(whi[k]); }
        const double padd = M * std::ldexp(1.0, -20);
        s->max_abs = M; s->dev.err_abs = (float)padd;
        // arena: what the render kernels read (nodes last: their number is known only after the build)
        size_t off = 0;
        auto place = [&](size_t bytes) { size_t o = off; off += (bytes + 255) & ~(size_t)255; return o; };
        const size_t n_items = n + 1;
        const size_t o_rank = place(lazy ? 0 : (size_t)8 * n_items * 4);
        const size_t o_s32 = place(ns * 16), o_s64 = place(ns * 32), o_smat = place(ns * 4), o_sid = place(ns * 4);
        const size_t o_c32 = place(ncb * 32), o_c64 = place(ncb * 48), o_cmat = place(ncb * 4), o_cid = place(ncb * 4);
        const size_t o_tri = place(nt * 48), o_nrm = place(any_normals ? nt * 36 : 0);
        const size_t o_mat = place(mats.size() * 8), o_lights = place(d->n_lights * 72);
        const size_t o_nodes = place(n * 64);
        const size_t arena_cap = off;
        // scratch: the caller's arrays as they are, the items, the builder's work space
        off = 0;
        const size_t r_sph = place(ns * sizeof(lgb_sphere)), r_smat = place(ns * 4), r_sid = place(ns * 4);
        const size_t r_cub = place(ncb * sizeof(lgb_cuboid)), r_cmat = place(ncb * 4), r_cid = place(ncb * 4);
        const size_t r_tri = place(nt * sizeof(lgb_triangle)), r_tmat = place(nt * 4), r_tid = place(nt * 4);
        const size_t r_nrm = place(any_normals ? nt * sizeof(lgb_tri_normals) : 0), r_has = place(any_normals && d->tri_has_normals ? nt : 0);
        const size_t raw_bytes = off;
        const size_t t_items = place(n * sizeof(GItem)), t_final = place(n * sizeof(GItem));
        const size_t build_bytes = gpu_build_temp_bytes((uint32_t)n);
        const size_t t_build = place(build_bytes);
        const size_t scratch_bytes = off;
        // pinned staging: [rank | materials | lights | raw arrays]
        const size_t st_rank = 0, st_mat = ((lazy ? 0 : (size_t)8 * n_items * 4) + 255) & ~(size_t)255, st_lights = st_mat + ((mats.size() * 8 + 255) & ~(size_t)255);
        const size_t st_raw = st_lights + ((d->n_lights * 72 + 255) & ~(size_t)255);
        void* scratch = nullptr;
        {
            cudaError_t e = ctx->reserve_staging(st_raw + raw_bytes);
            if (e != cudaSuccess) return bail(e == cudaErrorMemoryAllocation ? fail(ctx, LGB_ERR_NOMEM, "scene upload: pinned staging allocation failed") : cuda_fail(ctx, e, "cudaHostAlloc"));
            e = shared_alloc(ctx, &s->arena, arena_cap, ctx->stream);
            if (e != cudaSuccess) { s->arena = nullptr; return bail(e == cudaErrorMemoryAllocation ? fail(ctx, LGB_ERR_NOMEM, "scene upload: device allocation failed") : cuda_fail(ctx, e, "cudaMallocAsync")); }
            e = cudaMallocAsync(&scratch, scratch_bytes, ctx->stream);
            if (e != cudaSuccess) {
                size_t fr = 0, tot = 0; cudaGetLastError(); cudaMemGetInfo(&fr, &tot);
                char msg[160]; std::snprintf(msg, sizeof msg, "scene build: device scratch allocation of %zu bytes failed (%zu of %zu bytes free on the device)", scratch_bytes, fr, tot);
                return bail(e == cudaErrorMemoryAllocation ? fail(ctx, LGB_ERR_NOMEM, msg) : cuda_fail(ctx, e, "cudaMallocAsync"));
            }
        }
        char* H = (char*)ctx->staging; char* D = (char*)s->arena; char* T = (char*)scratch;
        auto gfail = [&](int code) { if (!s->deferred.scratch) cudaFreeAsync(scratch, ctx->stream); return bail(code); };
        Pool& pool = Pool::get();
        // the caller's arrays go through the pinned buffer in chunks: while one chunk crosses PCIe the host threads stage the next
        cudaError_t stage_err = cudaSuccess;
        auto stage = [&](size_t at, const void* src, size_t bytes) {
            constexpr size_t kChunk = 4u << 20;
            for (size_t c0 = 0; c0 < bytes && stage_err == cudaSuccess; c0 += kChunk) {
                const size_t len = std::min(kChunk, bytes - c0);
                pool.for_range(len, 256u << 10, [&](size_t b, size_t e, size_t) { std::memcpy(H + st_raw + at + c0 + b, (const char*)src + c0 + b, e - b); });
                stage_err = cudaMemcpyAsync(T + at + c0, H + st_raw + at + c0, len, cudaMemcpyHostToDevice, ctx->stream);
            }
        };
        stage(r_sph, d->spheres, ns * sizeof(lgb_sphere)); stage(r_smat, d->sphere_material, ns * 4); stage(r_sid, d->sphere_id, ns * 4);
        stage(r_cub, d->cuboids, ncb * sizeof(lgb_cuboid)); stage(r_cmat, d->cuboid_material, ncb * 4); stage(r_cid, d->cuboid_id, ncb * 4);
        stage(r_tri, d->triangles, nt * sizeof(lgb_triangle)); stage(r_tmat, d->triangle_material, nt * 4); stage(r_tid, d->triangle_id, nt * 4);
        if (any_normals) { stage(r_nrm, d->tri_normals, nt * sizeof(lgb_tri_normals)); if (d->tri_has_normals) stage(r_has, d->tri_has_normals, nt); }
        cudaError_t e = stage_err;
        if (e != cudaSuccess) { cuda_fail(ctx, e, "cudaMemcpyAsync(H2D raw scene)"); return gfail(LGB_ERR_CUDA); }
        RawScene raw{};
        raw.spheres = (const lgb_sphere*)(T + r_sph); raw.sphere_material = (const uint32_t*)(T + r_smat); raw.sphere_id = (const uint32_t*)(T + r_sid); raw.n_spheres = (uint32_t)ns;
        raw.cuboids = (const lgb_cuboid*)(T + r_cub); raw.cuboid_material = (const uint32_t*)(T + r_cmat); raw.cuboid_id = (const uint32_t*)(T + r_cid); raw.n_cuboids = (uint32_t)ncb;
        raw.triangles = (const lgb_triangle*)(T + r_tri); raw.triangle_material = (const uint32_t*)(T + r_tmat); raw.triangle_id = (const uint32_t*)(T + r_tid); raw.n_triangles = (uint32_t)nt;
        raw.tri_normals = any_normals ? (const lgb_tri_normals*)(T + r_nrm) : nullptr;
        raw.tri_has_normals = any_normals && d->tri_has_normals ? (const uint8_t*)(T + r_has) : nullptr;
        GItem* items = (GItem*)(T + t_items); GItem* final_items = (GItem*)(T + t_final);
        if ((e = launch_make_items(raw, (float)padd, items, ctx->stream)) != cudaSuccess) { cuda_fail(ctx, e, "k_make_items"); return gfail(LGB_ERR_CUDA); }
        s->t_validate = ms_since(tc0);
        // while the copy and the item kernel run: rank tables from the caller's reference tree, materials, lights
        auto tr0 = std::chrono::steady_clock::now();
        if (!lazy) {
            BuiltScene one; one.spaces.emplace_back(); one.inst_space.assign(d->n_instances, kNoSpace);
            if (!build_rank_tables(d, prim_count, one, (uint32_t*)(H + st_rank)))
                return gfail(fail(ctx, LGB_ERR_INVALID, "lgb_scene_create: primitive ids must be a permutation of 0..n-1 and every primitive must be referenced by exactly one leaf"));
        }
        std::memcpy(H + st_mat, mats.data(), mats.size() * 8);
        {
            double* l = (double*)(H + st_lights);
            for (uint64_t i = 0; i < d->n_lights; i++)
                for (int k = 0; k < 3; k++) { l[9 * i + k] = d->lights[i].position[k]; l[9 * i + 3 + k] = d->lights[i].intensity[k]; l[9 * i + 6 + k] = d->lights[i].falloff[k]; }
        }
        s->t_rank = ms_since(tr0);
        if ((!lazy && (e = cudaMemcpyAsync(D + o_rank, H + st_rank, (size_t)8 * n_items * 4, cudaMemcpyHostToDevice, ctx->stream)) != cudaSuccess) ||
            (e = cudaMemcpyAsync(D + o_mat, H + st_mat, mats.size() * 8, cudaMemcpyHostToDevice, ctx->stream)) != cudaSuccess ||
            (d->n_lights && (e = cudaMemcpyAsync(D + o_lights, H + st_lights, d->n_lights * 72, cudaMemcpyHostToDevice, ctx->stream)) != cudaSuccess)) {
            cuda_fail(ctx, e, "cudaMemcpyAsync(H2D)"); return gfail(LGB_ERR_CUDA);
        }
        auto tb0 = std::chrono::steady_clock::now();
        GpuBuildInfo info{};
        uint32_t* typepos[3] = {nullptr, nullptr, nullptr};
        LeafArrays la{};
        la.sph32 = (float4*)(D + o_s32); la.sph64 = (double*)(D + o_s64); la.sph_mat = (uint32_t*)(D + o_smat); la.sph_id = (uint32_t*)(D + o_sid);
        la.cub32 = (float4*)(D + o_c32); la.cub64 = (double*)(D + o_c64); la.cub_mat = (uint32_t*)(D + o_cmat); la.cub_id = (uint32_t*)(D + o_cid);
        la.tri = (float4*)(D + o_tri); la.tri_nrm = any_normals ? (float*)(D + o_nrm) : nullptr;
        // plastic scenes whose shadow rays will have light grids: no tree yet (see lgb_scene::Deferred); everything else builds it now
        // ... and whose primary rays will have a camera grid: known only if the caller says how large the film is (the grid pays from four
        // samples per primitive, ensure_camgrid); LGB_OPT_LAZY_BVH = 1 defers regardless
        const uint64_t expect_samples = (uint64_t)d->expected_film_pixels * d->camera.supersampling_root * d->camera.supersampling_root;
        const bool cam_grid_likely = d->camera.pixel_separation == 0.0 && ctx->camera_grid != 0 && (ctx->camera_grid == 1 || expect_samples >= 4ull * n);
        const bool grids_likely = ctx->light_grids == 1 || (ctx->light_grids < 0 && d->n_lights <= 8 && !(expect_samples && expect_samples * d->n_lights < 8ull * n));
        const bool defer = (ctx->lazy_bvh == 1 || (ctx->lazy_bvh < 0 && cam_grid_likely)) && !any_general && d->n_lights >= 1 && grids_likely;
        if (defer) {
            if ((e = gpu_identity_positions(items, (uint32_t)n, typepos, T + t_build, build_bytes, ctx->stream)) != cudaSuccess) { cuda_fail(ctx, e, "gpu_identity_positions"); return gfail(LGB_ERR_CUDA); }
            if ((e = launch_convert(raw, la, items, (uint32_t)n, typepos, padd, ctx->stream)) != cudaSuccess) { cuda_fail(ctx, e, "k_convert"); return gfail(LGB_ERR_CUDA); }
            s->deferred.scratch = scratch; s->deferred.raw = raw; s->deferred.items = items; s->deferred.final_items = final_items; s->deferred.la = la;
            s->deferred.build_temp = T + t_build; s->deferred.build_bytes = build_bytes; s->deferred.o_nodes = o_nodes; s->deferred.n = (uint32_t)n; s->deferred.padd = padd;
        } else {
            e = gpu_build_sah(items, (uint32_t)n, (HostNode*)(D + o_nodes), final_items, typepos, T + t_build, build_bytes, ctx->stream, &info);
            if (e != cudaSuccess) { cuda_fail(ctx, e, "gpu_build_sah"); return gfail(LGB_ERR_CUDA); }
            if (info.max_depth + 1 > (uint32_t)kStackDepth) return gfail(fail(ctx, LGB_ERR_UNSUPPORTED, "device BVH deeper than the 64-entry traversal stack"));
            if ((e = launch_convert(raw, la, final_items, (uint32_t)n, typepos, padd, ctx->stream)) != cudaSuccess) { cuda_fail(ctx, e, "k_convert"); return gfail(LGB_ERR_CUDA); }
            cudaFreeAsync(scratch, ctx->stream);
        }
        s->build_ms = ms_since(tb0);
        s->t_build = s->build_ms;
        s->bytes = o_nodes + (size_t)info.n_nodes * 64;
        s->dev.nodes = defer ? nullptr : (const float4*)(D + o_nodes); s->dev.n_nodes = info.n_nodes;
        s->dev.rank = lazy ? nullptr : (const uint32_t*)(D + o_rank); s->dev.prim_count = prim_count; s->dev.rank_items = (uint32_t)n_items;
        s->dev.n_sph = (uint32_t)ns; s->dev.n_cub = (uint32_t)ncb; s->dev.n_tri = (uint32_t)nt;
        s->dev.n_spaces = 1; s->dev.instanced = 0;
        if (lazy) { s->lazy_fn = d->reference_tree; s->lazy_user = d->reference_tree_user; s->lazy_desc = *d; }
        if (ns) { s->dev.sph32 = la.sph32; s->dev.sph64 = la.sph64; s->dev.sph_mat = la.sph_mat; s->dev.sph_id = la.sph_id; }
        if (ncb) { s->dev.cub32 = la.cub32; s->dev.cub64 = la.cub64; s->dev.cub_mat = la.cub_mat; s->dev.cub_id = la.cub_id; }
        if (nt) { s->dev.tri = la.tri; s->dev.tri_nrm = la.tri_nrm; }
        s->dev.materials = (const double*)(D + o_mat);
        s->dev.lights = d->n_lights ? (const double*)(D + o_lights) : nullptr; s->dev.n_lights = (uint32_t)d->n_lights;
        s->dev.general = any_general; s->dev.specular = any_specular; s->dev.recursion = d->recursion;
        s->gpu_built = true;
        (void)tg0;
    } else {
    auto tc2 = std::chrono::steady_clock::now();
    BuiltScene bvh;
    {
        std::string berr;
        const int brc = build_scene(d, wlo, whi, bvh, berr);
        if (brc == -2 || brc == -4) return bail(fail(ctx, LGB_ERR_UNSUPPORTED, "lgb_scene_create: " + berr));
        if (brc) return bail(fail(ctx, LGB_ERR_INVALID, "lgb_scene_create: " + berr));
        if (bvh.spaces[0].stack_need > (uint32_t)kStackDepth) return bail(fail(ctx, LGB_ERR_UNSUPPORTED, "device BVH deeper than the 64-entry traversal stack"));
        if (bvh.spaces.size() > 1) for (const HostSpace& sp : bvh.spaces) if (sp.depth >= (uint32_t)kMaxSpaceDepth) return bail(fail(ctx, LGB_ERR_UNSUPPORTED, "more than 8 nested transformed aggregates"));
    }
    const double padd = bvh.spaces[0].max_abs * std::ldexp(1.0, -20);
    s->max_abs = bvh.spaces[0].max_abs;
    s->dev.err_abs = bvh.spaces[0].err_abs;
    const bool instanced = bvh.instanced();
    const size_t nsp = bvh.spaces.size();
    s->build_ms = bvh.build_ms;
    s->t_build = ms_since(tc2);

    // ---- layout of the scene arena: every array at a 256-byte aligned offset of ONE allocation, assembled in
    //      pinned host memory by all threads and moved with one H2D copy
    static_assert(sizeof(HostNode) == 64, "node layout");
    const size_t ns = d->n_spheres, ncb = d->n_cuboids, nt = d->n_triangles, nnodes = bvh.nodes.size();
    const bool any_normals = nt && d->tri_normals;
    size_t off = 0;
    auto place = [&](size_t bytes) { size_t o = off; off += (bytes + 255) & ~(size_t)255; return o; };
    const size_t n_items = (size_t)prim_count + nsp;       // rank-table items: primitives, then one per space
    const size_t o_nodes = place(nnodes * 64), o_rank = place((size_t)8 * n_items * 4);
    const size_t o_spaces = place(instanced ? nsp * sizeof(DevSpace) : 0), o_inst = place(instanced ? bvh.order[3].size() * 4 : 0);
    const size_t o_sspace = place(instanced ? ns * 4 : 0), o_cspace = place(instanced ? ncb * 4 : 0), o_tspace = place(instanced ? nt * 4 : 0);
    const size_t o_s32 = place(ns * 16), o_s64 = place(ns * 32), o_smat = place(ns * 4), o_sid = place(ns * 4);
    const size_t o_c32 = place(ncb * 32), o_c64 = place(ncb * 48), o_cmat = place(ncb * 4), o_cid = place(ncb * 4);
    const size_t o_tri = place(nt * 48), o_nrm = place(any_normals ? nt * 36 : 0);
    const size_t o_mat = place(mats.size() * 8), o_lights = place(d->n_lights * 72);
    const size_t arena_bytes = off;
    {
        cudaError_t e = ctx->reserve_staging(arena_bytes);
        if (e != cudaSuccess) return bail(e == cudaErrorMemoryAllocation ? fail(ctx, LGB_ERR_NOMEM, "scene upload: pinned staging allocation failed") : cuda_fail(ctx, e, "cudaHostAlloc"));
        e = shared_alloc(ctx, &s->arena, arena_bytes, ctx->stream);
        if (e != cudaSuccess) { s->arena = nullptr; return bail(e == cudaErrorMemoryAllocation ? fail(ctx, LGB_ERR_NOMEM, "scene upload: device allocation failed") : cuda_fail(ctx, e, "cudaMallocAsync")); }
        s->bytes = arena_bytes;
        // the previous scene's H2D copy out of the staging buffer is complete: lgb_scene_create synchronises before returning
    }
    char* H = (char*)ctx->staging;
    char* D = (char*)s->arena;
    auto tc1 = std::chrono::steady_clock::now();
    (void)threads;
    if (!build_rank_tables(d, prim_count, bvh, (uint32_t*)(H + o_rank)))
        return bail(fail(ctx, LGB_ERR_INVALID, "lgb_scene_create: primitive ids must be a permutation of 0..n-1 and every primitive must be referenced by exactly one leaf"));
    s->t_rank = ms_since(tc1);
    auto tc3 = std::chrono::steady_clock::now();
    Pool& pool = Pool::get();
    pool.for_range(nnodes, 1 << 14, [&](size_t b, size_t e, size_t) { std::memcpy(H + o_nodes + b * 64, bvh.nodes.data() + b, (e - b) * 64); });
    s->dev.nodes = (const float4*)(D + o_nodes); s->dev.n_nodes = (uint32_t)nnodes;
    s->dev.rank = (const uint32_t*)(D + o_rank); s->dev.prim_count = prim_count; s->dev.rank_items = (uint32_t)n_items;
    s->dev.n_sph = (uint32_t)ns; s->dev.n_cub = (uint32_t)ncb; s->dev.n_tri = (uint32_t)nt;
    s->dev.n_spaces = (uint32_t)nsp; s->dev.instanced = instanced ? 1u : 0u;
    if (instanced) {
        DevSpace* ds = (DevSpace*)(H + o_spaces);
        for (size_t k = 0; k < nsp; k++) {
            const HostSpace& sp = bvh.spaces[k];
            std::memcpy(ds[k].m, sp.m, sizeof sp.m); std::memcpy(ds[k].minv, sp.minv, sizeof sp.minv);
            ds[k].parent = sp.parent; ds[k].depth = sp.depth; ds[k].root_node = sp.root_node;
            ds[k].flags = (sp.identity ? kSpaceIdentity : 0u) | (sp.swap_backface ? kSpaceSwap : 0u);
            ds[k].err_abs = sp.err_abs; ds[k].pad[0] = ds[k].pad[1] = ds[k].pad[2] = 0;
        }
        std::memcpy(H + o_inst, bvh.order[3].data(), bvh.order[3].size() * 4);
        s->dev.spaces = (const DevSpace*)(D + o_spaces); s->dev.inst_space = (const uint32_t*)(D + o_inst);
        s->dev.sph_space = (const uint32_t*)(D + o_sspace); s->dev.cub_space = (const uint32_t*)(D + o_cspace); s->dev.tri_space = (const uint32_t*)(D + o_tspace);
    }
    if (ns) {
        const uint32_t* ord = bvh.order[LGB_PRIM_SPHERE].data();
        float4* s32 = (float4*)(H + o_s32); double* s64 = (double*)(H + o_s64); uint32_t* m = (uint32_t*)(H + o_smat); uint32_t* id = (uint32_t*)(H + o_sid);
        pool.for_range(ns, 1 << 14, [&](size_t b, size_t e, size_t) {
            for (size_t j = b; j < e; j++) {
                const uint32_t i = ord[j];
                const lgb_sphere& sp = d->spheres[i];
                s32[j] = make_float4((float)sp.center[0], (float)sp.center[1], (float)sp.center[2], f32_up(std::fabs(sp.radius)));
                s64[4 * j] = sp.center[0]; s64[4 * j + 1] = sp.center[1]; s64[4 * j + 2] = sp.center[2]; s64[4 * j + 3] = sp.radius;
                m[j] = d->sphere_material[i]; id[j] = d->sphere_id[i];
                if (instanced) ((uint32_t*)(H + o_sspace))[j] = bvh.prim_space[0].empty() ? 0u : bvh.prim_space[0][i];
            }
        });
        s->dev.sph32 = (const float4*)(D + o_s32); s->dev.sph64 = (const double*)(D + o_s64);
        s->dev.sph_mat = (const uint32_t*)(D + o_smat); s->dev.sph_id = (const uint32_t*)(D + o_sid);
    }
    if (ncb) {
        const uint32_t* ord = bvh.order[LGB_PRIM_CUBOID].data();
        float4* c32 = (float4*)(H + o_c32); double* c64 = (double*)(H + o_c64); uint32_t* m = (uint32_t*)(H + o_cmat); uint32_t* id = (uint32_t*)(H + o_cid);
        pool.for_range(ncb, 1 << 14, [&](size_t b, size_t e, size_t) {
            for (size_t j = b; j < e; j++) {
                const uint32_t i = ord[j];
                const lgb_cuboid& c = d->cuboids[i];
                const uint32_t spc = bvh.prim_space[1].empty() ? 0u : bvh.prim_space[1][i];
                const double pad = bvh.spaces[spc].max_abs * std::ldexp(1.0, -20);
                c32[2 * j] = make_float4(f32_down(c.min[0] - pad), f32_down(c.min[1] - pad), f32_down(c.min[2] - pad), 0.f);
                c32[2 * j + 1] = make_float4(f32_up(c.max[0] + pad), f32_up(c.max[1] + pad), f32_up(c.max[2] + pad), 0.f);
                if (instanced) ((uint32_t*)(H + o_cspace))[j] = spc;
                for (int k = 0; k < 3; k++) { c64[6 * j + k] = c.min[k]; c64[6 * j + 3 + k] = c.max[k]; }
                m[j] = d->cuboid_material[i]; id[j] = d->cuboid_id[i];
            }
        });
        s->dev.cub32 = (const float4*)(D + o_c32); s->dev.cub64 = (const double*)(D + o_c64);
        s->dev.cub_mat = (const uint32_t*)(D + o_cmat); s->dev.cub_id = (const uint32_t*)(D + o_cid);
    }
    if (nt) {
        const uint32_t* ord = bvh.order[LGB_PRIM_TRIANGLE].data();
        float4* t = (float4*)(H + o_tri); float* nrm = (float*)(H + o_nrm);
        pool.for_range(nt, 1 << 14, [&](size_t b0, size_t e0, size_t) {
            for (size_t j = b0; j < e0; j++) {
                const uint32_t i = ord[j];
                const lgb_triangle& tr = d->triangles[i];
                uint32_t ni = kNoNormals;
                if (any_normals && (!d->tri_has_normals || d->tri_has_normals[i])) {      // normals slot j (leaf order)
                    ni = (uint32_t)j;
                    const lgb_tri_normals& q = d->tri_normals[i];
                    float* o = nrm + 9 * j;
                    for (int k = 0; k < 3; k++) { o[k] = q.n0[k]; o[3 + k] = q.n1[k]; o[6 + k] = q.n2[k]; }
                } else if (any_normals) std::memset(nrm + 9 * j, 0, 36);
                float4 a = make_float4(tr.p0[0], tr.p0[1], tr.p0[2], 0.f), b = make_float4(tr.p1[0], tr.p1[1], tr.p1[2], 0.f), c = make_float4(tr.p2[0], tr.p2[1], tr.p2[2], 0.f);
                std::memcpy(&a.w, &d->triangle_id[i], 4); std::memcpy(&b.w, &d->triangle_material[i], 4); std::memcpy(&c.w, &ni, 4);
                t[3 * j] = a; t[3 * j + 1] = b; t[3 * j + 2] = c;
                if (instanced) ((uint32_t*)(H + o_tspace))[j] = bvh.prim_space[2].empty() ? 0u : bvh.prim_space[2][i];
            }
        });
        s->dev.tri = (const float4*)(D + o_tri);
        s->dev.tri_nrm = any_normals ? (const float*)(D + o_nrm) : nullptr;
    }
    std::memcpy(H + o_mat, mats.data(), mats.size() * 8);
    s->dev.materials = (const double*)(D + o_mat);
    {
        double* l = (double*)(H + o_lights);
        for (uint64_t i = 0; i < d->n_lights; i++)
            for (int k = 0; k < 3; k++) { l[9 * i + k] = d->lights[i].position[k]; l[9 * i + 3 + k] = d->lights[i].intensity[k]; l[9 * i + 6 + k] = d->lights[i].falloff[k]; }
        s->dev.lights = d->n_lights ? (const double*)(D + o_lights) : nullptr;      // (an empty array at the very end of the arena has no valid offset)
        s->dev.n_lights = (uint32_t)d->n_lights;
        s->dev.general = any_general; s->dev.specular = any_specular; s->dev.recursion = d->recursion;
    }
    {
        cudaError_t e = cudaMemcpyAsync(D, H, arena_bytes, cudaMemcpyHostToDevice, ctx->stream);
        if (e != cudaSuccess) { cuda_fail(ctx, e, "cudaMemcpyAsync(H2D)"); return bail(LGB_ERR_CUDA); }
    }
    s->t_convert_upload = ms_since(tc3);
    }
    for (int k = 0; k < 3; k++) {
        s->cam.origin[k] = d->camera.origin[k]; s->cam.view[k] = d->camera.view[k]; s->cam.up[k] = d->camera.up[k]; s->cam.aux[k] = d->camera.aux[k];
        s->shade.ambient[k] = d->ambient[k]; s->shade.bg_inner[k] = d->bg_inner[k]; s->shade.bg_outer[k] = d->bg_outer[k];
    }
    s->cam.image_plane_height = d->camera.image_plane_height;
    s->cam.pixel_separation = d->camera.pixel_separation;
    s->cam.sample_distance = d->camera.sample_distance;
    s->cam.root = d->camera.supersampling_root;
    s->shade.bg_scale = d->bg_scale;
    cudaError_t e = cudaStreamSynchronize(ctx->stream);     // the staging buffer is free for the next scene
    if (e != cudaSuccess) { cuda_fail(ctx, e, "scene upload"); return bail(LGB_ERR_CUDA); }
    s->t_total = ms_since(tc0);
    if (getenv("LGB_TIMING")) fprintf(stderr, "[lgb_scene_create] %s build: validate%s %.1f rank %.1f build %.1f (sah %.1f) convert+upload %.1f total %.1f ms, %u threads\n",
                                      s->gpu_built ? "device" : "host", s->gpu_built ? "+stage" : "", s->t_validate, s->t_rank, s->t_build, s->build_ms, s->t_convert_upload, s->t_total, (unsigned)threads);
    if (ctx->peers.empty()) { if (int rc = build_light_grids(ctx, s)) return bail(rc); }
    else if (int rc = replicate_to_peers(ctx, s)) return bail(rc);       // (builds the leader's grids too, while the peers copy)
    *out = s;
    return LGB_OK;
}

// ---------------------------------------------------------------------------------------- capture
// Macro tiles are dealt to ranks round-robin along anti-diagonals: owner = (mx + my) % ranks.
static void build_tile_list(lgb_ctx* c, uint32_t w, uint32_t h, uint32_t rank, uint32_t ranks) {
    if (c->tile_key[0] == w && c->tile_key[1] == h && c->tile_key[2] == rank && c->tile_key[3] == ranks && c->tile_count) return;
    const uint32_t nmx = (w + kMacroTile - 1) / kMacroTile, nmy = (h + kMacroTile - 1) / kMacroTile;
    c->tile_host.clear();
    for (uint32_t my = 0; my < nmy; my++)
        for (uint32_t mx = 0; mx < nmx; mx++)
            if ((mx + my) % ranks == rank) c->tile_host.push_back(my * nmx + mx);
    c->tile_key[0] = w; c->tile_key[1] = h; c->tile_key[2] = rank; c->tile_key[3] = ranks;
    c->tile_count = 0;   // uploaded lazily
}

// Camera grid of `s` for a w x h film (lgb_grid.cu), built on first use and kept with the scene; fills W.cg_* or leaves them NULL
// (orthographic camera, transformed aggregates, a scene too small to pay for the binning, too many primitives across the eye's plane).
static int ensure_camgrid(lgb_ctx* c, lgb_scene* s, uint32_t w, uint32_t h, uint64_t samples, DevWork& W, cudaStream_t st) {
    const DevScene& S = s->dev;
    const uint32_t prims = S.n_sph + S.n_cub + S.n_tri;
    // automatic: where the frame holds enough samples to pay for binning every primitive (measured, DESIGN.md)
    const bool want = c->camera_grid == 1 || (c->camera_grid < 0 && large_scene(S) && samples >= 4ull * prims);
    if (!want || S.instanced || s->cam.pixel_separation != 0.0 || prims == 0) return LGB_OK;
    lgb_scene::CamGrid& G = s->cam_grid();
    if (G.refused && G.w == w && G.h == h) return LGB_OK;
    if (!(G.valid && G.w == w && G.h == h)) {
        auto t0 = std::chrono::steady_clock::now();
        for (void** q : {&G.starts, &G.entries, &G.large}) if (*q) { cudaFreeAsync(*q, st); *q = nullptr; }
        G.valid = false; G.refused = false; G.w = w; G.h = h;
        CamGridParams P{};
        const DevCamera& cam = s->cam;
        // (a w, b w, w) = [aux | up | view]^-1 (X - origin)
        const double m[9] = {cam.aux[0], cam.up[0], cam.view[0], cam.aux[1], cam.up[1], cam.view[1], cam.aux[2], cam.up[2], cam.view[2]};
        const double det = m[0] * (m[4] * m[8] - m[5] * m[7]) - m[1] * (m[3] * m[8] - m[5] * m[6]) + m[2] * (m[3] * m[7] - m[4] * m[6]);
        if (!(std::fabs(det) > 1e-300) || !std::isfinite(det)) { G.refused = true; return LGB_OK; }
        const double id = 1.0 / det;
        P.minv[0] = (m[4] * m[8] - m[5] * m[7]) * id; P.minv[1] = (m[2] * m[7] - m[1] * m[8]) * id; P.minv[2] = (m[1] * m[5] - m[2] * m[4]) * id;
        P.minv[3] = (m[5] * m[6] - m[3] * m[8]) * id; P.minv[4] = (m[0] * m[8] - m[2] * m[6]) * id; P.minv[5] = (m[2] * m[3] - m[0] * m[5]) * id;
        P.minv[6] = (m[3] * m[7] - m[4] * m[6]) * id; P.minv[7] = (m[1] * m[6] - m[0] * m[7]) * id; P.minv[8] = (m[0] * m[4] - m[1] * m[3]) * id;
        for (int k = 0; k < 3; k++) P.origin[k] = cam.origin[k];
        P.iph = cam.image_plane_height; P.ipw = cam.image_plane_height * ((double)w / (double)h); P.w = (double)w; P.h = (double)h;
        if (!(P.iph != 0.0) || !std::isfinite(P.iph)) { G.refused = true; return LGB_OK; }
        P.delta0 = std::min(0.5 * cam.sample_distance, (cam.root - 0.5) * cam.sample_distance);
        P.delta1 = std::max(0.5 * cam.sample_distance, (cam.root - 0.5) * cam.sample_distance);
        P.w_eps = 1e-6;
        P.shift = 2;
        if (const char* e = std::getenv("LGB_CAM_SHIFT")) P.shift = std::min(6, std::max(0, std::atoi(e)));
        P.nx = ((w - 1) >> P.shift) + 1; P.ny = ((h - 1) >> P.shift) + 1;
        P.large_cells = kGridLargeCells; P.large_cap = kGridLargeCap;
        const size_t nc = (size_t)P.nx * P.ny, scan_bytes = scan_bytes_for(nc);
        auto up = [](size_t v) { return (v + 255) & ~(size_t)255; };
        char* tmp_a = nullptr;                                   // counts | scan scratch | large counter: one allocation (see build_light_grids)
        CU(c, cudaMallocAsync((void**)&tmp_a, up((nc + 1) * 4) + up(std::max<size_t>(scan_bytes, 16)) + 256, st));
        uint32_t* counts = (uint32_t*)tmp_a; void* scan_tmp = tmp_a + up((nc + 1) * 4); uint32_t* n_large_dev = (uint32_t*)(tmp_a + up((nc + 1) * 4) + up(std::max<size_t>(scan_bytes, 16)));
        CU(c, cudaMallocAsync(&G.starts, (nc + 1) * 4, st));
        CU(c, cudaMallocAsync(&G.large, sizeof(uint2) * kGridLargeCap, st));
        uint32_t total = 0, n_large = 0;
        CU(c, camgrid_count(S, P, counts, (uint32_t*)G.starts, scan_tmp, scan_bytes, (uint2*)G.large, n_large_dev, st, &total, &n_large));
        if (n_large > kGridLargeCap) G.refused = true;
        else {
            char* tmp_b = nullptr;                               // unsorted entries | sort scratch
            const size_t sort_bytes = grid_sort_bytes(total, nc), b_entries = up(sizeof(uint2) * std::max<size_t>(total, 1));
            CU(c, cudaMallocAsync(&G.entries, sizeof(uint2) * std::max<size_t>(total, 1), st));
            CU(c, cudaMallocAsync((void**)&tmp_b, b_entries + std::max<size_t>(sort_bytes, 16), st));
            void* entries_tmp = tmp_b; void* sort_tmp = tmp_b + b_entries;
            CU(c, camgrid_fill(S, P, counts, (const uint32_t*)G.starts, (uint2*)entries_tmp, (uint2*)G.entries, total, sort_tmp, sort_bytes, (uint2*)G.large, n_large, st));
            cudaFreeAsync(tmp_b, st);
            G.valid = true; G.shift = P.shift; G.nx = P.nx; G.n_large = n_large; G.bytes = (nc + 1) * 4 + sizeof(uint2) * ((size_t)total + n_large);
        }
        cudaFreeAsync(tmp_a, st);
        G.build_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
        if (getenv("LGB_TIMING")) fprintf(stderr, "[camera grid] %ux%u tiles of %u px: %u entries, %u large, %.2f ms (host clock, incl. one sync)%s\n", P.nx, P.ny, 1u << P.shift, total, n_large, G.build_ms, G.refused ? " REFUSED" : "");
    }
    if (G.valid) { W.cg_start = (const uint32_t*)G.starts; W.cg_entries = (const uint2*)G.entries; W.cg_large = (const uint2*)G.large; W.cg_n_large = G.n_large; W.cg_shift = G.shift; W.cg_nx = G.nx; }
    return LGB_OK;
}

// DevScene::self: the scene record in global memory for the launches queued on `st` from here on (out-of-line device functions read
// it there).  The source is pageable, so the record is taken before the call returns; whatever changes s->dev later -- rank tables,
// a deferred BVH -- comes back through here before it launches anything.
static int sync_scene_copy(lgb_ctx* c, lgb_scene* s, cudaStream_t st) {
    CU(c, c->scene_copy.reserve(sizeof(DevScene)));
    s->dev.self = (const DevScene*)c->scene_copy.p;
    CU(c, cudaMemcpyAsync(c->scene_copy.p, &s->dev, sizeof(DevScene), cudaMemcpyHostToDevice, st));
    return LGB_OK;
}

struct CaptureArgs {
    uint32_t w, h;
    uint32_t mode;               // 0 tiles, 1 stride subset
    uint32_t rank, ranks, k, n;
    bool aov;
    void* d_film;                // device film or NULL (context film)
    cudaStream_t stream;
    bool want_li = false;        // aov: also the radiance of every sample
    bool klog_no_camgrid = false;
    void* host_film = nullptr;   // lgb_capture: the caller's film; where the frame allows it the read-back starts behind the first slice of the shade kernel
    KernelLog* klog = nullptr;   // lgb_capture_profile: events and counter snapshots around every launch (one stream)
};

// Wavefront buffers of `nslots` sample slots carved out of one allocation (layout: DevWave, lgb_types.cuh).
static uint64_t fastdiv_magic(uint64_t d) { return d <= 1 ? 0ull : (~0ull) / d + 1ull; }      // fdiv(), lgb_kernels.cu
static void set_divisors(DevWork& W, uint32_t root) { W.fd_spp = fastdiv_magic(W.spp); W.fd_root = fastdiv_magic(root); W.fd_nmx = fastdiv_magic(W.n_macro_x); }
// camera.rs:115-118,131-133 once per launch (DevWork.cam_*): same operations, same order, IEEE doubles (this file is compiled without
// floating-point contraction), so the bits are the ones every thread used to compute for itself
static void set_camera_constants(DevWork& W, const DevCamera& C) {
    const double iph = C.image_plane_height;
    W.cam_ipw = iph * W.aspect;
    const double pixel_size = iph * W.hinv;
    const double sep = C.sample_distance * pixel_size;
    for (int k = 0; k < 3; k++) { W.cam_updiff[k] = C.up[k] * sep; W.cam_auxdiff[k] = C.aux[k] * sep; }
    for (int k = 0; k < 3; k++) W.cam_halfdiff[k] = W.cam_updiff[k] * 0.5 + W.cam_auxdiff[k] * 0.5;
}
static size_t wave_bytes(uint64_t nslots, uint32_t nl, uint64_t npix) { return nslots * (8 + 24 + 4 + 4 + 4 + 12 * (size_t)nl) + ((npix * 4 * nl + 15) & ~(uint64_t)15) + ((nslots + 15) & ~(uint64_t)15); }
static DevWave carve_wave(void* wave, void* ctr, uint64_t nslots, uint32_t nl, uint64_t npix = 1) {
    DevWave V{};
    char* base = (char*)wave;
    V.hit_t = (double*)base; base += nslots * 8;
    V.ps = (double*)base; base += nslots * 24;
    V.hit_ref = (uint32_t*)base; base += nslots * 4;
    V.occl = (uint32_t*)base; base += nslots * 4;
    V.gate = (uint32_t*)base; base += nslots * 4;
    V.queue = (uint32_t*)base; V.queue_stride = nslots; base += nslots * 12 * nl;
    V.occluder = (uint32_t*)base; base += (npix * 4 * nl + 15) & ~(uint64_t)15;
    V.sflags = (unsigned char*)base;
    V.work_counter = (unsigned long long*)ctr;
    V.queue_count = (uint32_t*)((char*)ctr + 8);
    V.queue_fetch = V.queue_count + LGB_MAX_LIGHTS * 3;
    V.tie_count = V.queue_fetch + LGB_MAX_LIGHTS * 3;
    V.fallback_count = V.tie_count + 1;
    V.sec_count = V.fallback_count + 1;
    V.free_count = V.sec_count + 2;
    V.fallback_list = V.queue;                       // the shadow queues are written only after the primary phase ...
    V.sec_list = V.queue;                            // ... and drained before k_shade lists the specular slots
    return V;
}

// Whitted recursion below the specular hits of the camera wave (integrate.rs:69-132), level by level.  k_shade of a wave has
// already turned its specular hits into the rays of the next level (spawn_children); here each level is traced and shaded with the
// RAYBUF variants of the frame's own kernels, and when a level spawns nothing (or scene.recursion is reached) the radiance is
// folded back up (k_gather).  One small device-to-host read per level sizes the next buffers and launches.
// prepare_spawn points wave `level` (slots sample slots) at the buffers of level + 1; false: not enough memory, use k_secondary.
static bool prepare_spawn(lgb_ctx* c, DevWave& V, uint32_t level, uint64_t slots) {
    if (c->lvl_recs[level].reserve((size_t)slots * sizeof(SpawnRec)) != cudaSuccess || c->raybuf[(level + 1) & 1].reserve(2 * (size_t)slots * 48) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    V.recs = (SpawnRec*)c->lvl_recs[level].p; V.next_rays = (double*)c->raybuf[(level + 1) & 1].p;
    V.spawn_ctr = (uint32_t*)c->lvl_ctr.p + 4 * level; V.next_t_base = (uint32_t)slots;
    return true;
}
static int run_whitted_levels(lgb_ctx* c, lgb_scene* s, const DevOut& O0, uint64_t slots0, cudaStream_t st, bool count, uint64_t* rays_traced, uint32_t* launches) {
    const DevScene& S = s->dev;
    const uint32_t nl = std::max<uint32_t>(S.n_lights, 1);
    const uint32_t* d_ctr = (const uint32_t*)c->lvl_ctr.p;
    uint64_t slots[kMaxRecursion + 2] = {slots0};    // sample slots of every level (holes included)
    int traced = 0;                                  // levels 1 .. traced exist
    std::vector<unsigned char> hctr(kWaveCtrBytes);
    for (uint32_t l = 0; l < S.recursion; l++) {
        uint32_t sc[4];                              // what wave l spawned: records, reflected rays, transmitted rays
        CU(c, cudaMemcpyAsync(sc, d_ctr + 4 * l, 16, cudaMemcpyDeviceToHost, st));
        CU(c, cudaStreamSynchronize(st));
        const uint64_t n_r = sc[1], n_t = sc[2];
        if (n_r + n_t == 0) break;
        const uint64_t n = n_t ? slots[l] + n_t : n_r;               // reflected rays from slot 0, transmitted ones from slots[l]
        if (n >= (1ull << 32) - 64) return fail(c, LGB_ERR_UNSUPPORTED, "capture: more than 2^32 rays in one level of the specular ray trees");
        slots[l + 1] = n; traced = (int)l + 1;
        CU(c, c->lvl_rad[l + 1].reserve((size_t)n * 24));
        CU(c, c->wave2.reserve(wave_bytes(n, nl, 1)));
        CU(c, c->wave2_ctr.reserve(kWaveCtrBytes));
        DevWork Wl{};
        Wl.mode = 3; Wl.w = (uint32_t)n; Wl.h = 1; Wl.n_pixels = n; Wl.spp = 1; Wl.rays = (const double*)c->raybuf[(l + 1) & 1].p; Wl.depth = l + 1;
        Wl.hole_lo = (uint32_t)n_r; Wl.hole_hi = n_t ? (uint32_t)slots[l] : (uint32_t)n_r;
        set_divisors(Wl, 1);
        DevWave Vl = carve_wave(c->wave2.p, c->wave2_ctr.p, n, nl);
        if (l + 1 < S.recursion && !prepare_spawn(c, Vl, l + 1, n)) return fail(c, LGB_ERR_CUDA, "capture: out of device memory for a level of the specular ray trees");
        DevOut Ol{}; Ol.radiance = (double*)c->lvl_rad[l + 1].p;
        CU(c, launch_level(S, s->cam, s->shade, Wl, Ol, Vl, c->sm_count, st, count ? (DevCounters*)c->counters.p : nullptr));
        *launches += 4 + (S.grids ? 1 : S.n_lights);                 // k_primary, k_setup, k_shadow x lights (or k_gshadow), k_shade; k_gather on the way back
        *rays_traced += n_r + n_t;
        if (count) {                                                 // + the shadow rays of this level (lgb_stats.secondary_rays)
            CU(c, cudaMemcpyAsync(hctr.data(), c->wave2_ctr.p, kWaveCtrBytes, cudaMemcpyDeviceToHost, st));
            CU(c, cudaStreamSynchronize(st));
            const uint32_t* qc = (const uint32_t*)(hctr.data() + 8);
            for (uint32_t k = 0; k < S.n_lights; k++) *rays_traced += qc[k * 3 + kQueueA];
        }
    }
    for (int l = traced - 1; l >= 0; l--)
        CU(c, launch_gather((const SpawnRec*)c->lvl_recs[l].p, d_ctr + 4 * l, l == 0 ? O0.radiance : (double*)c->lvl_rad[l].p, (const double*)c->lvl_rad[l + 1].p, slots[l], st));
    return LGB_OK;
}

// One frame (or this rank's tiles of it, or a stride subset).  The per-sample wavefront buffers are sized for a BAND of the work --
// as many macro tiles (or subset pixels) as fit the context's memory budget (LGB_OPT_WAVE_BUDGET_MB, default 16 GiB; a band also
// stays below 2^32 sample slots, which the kernels index with 32 bits) -- and the kernel sequence runs band after band on the same
// buffers: a frame of any size renders in bounded memory (8K at 64 spp: 2.1 G samples), and `mixed4k` is one band.
static int run_capture(lgb_ctx* c, lgb_scene* s, const CaptureArgs& a, lgb_stats* stats, bool sync_stats) {
    if (!c || !s || s->ctx != c) return fail(c, LGB_ERR_INVALID, "capture: scene does not belong to this context");
    if (a.w == 0 || a.h == 0 || (uint64_t)a.w * a.h >= (1ull << 32)) return fail(c, LGB_ERR_INVALID, "capture: bad film size");
    CU(c, cudaSetDevice(c->device));
    cudaStream_t st = a.stream ? a.stream : c->stream;
    DevWork W{};
    W.mode = a.mode; W.w = a.w; W.h = a.h;
    W.winv = 1.0 / (double)a.w; W.hinv = 1.0 / (double)a.h; W.aspect = (double)a.w / (double)a.h;   // film.rs:36-45
    W.spp = s->cam.root * s->cam.root;
    W.anchor = (s->cam.root / 2) * s->cam.root + s->cam.root / 2;      // camera.rs:143: sample (i, j) = i * root + j
    const uint64_t area = (uint64_t)a.w * a.h;
    uint64_t units_all = 0;                      // macro tiles (mode 0) or pixels (mode 1) of this call
    if (a.mode == 0) {
        if (a.ranks == 0 || a.rank >= a.ranks) return fail(c, LGB_ERR_INVALID, "capture: tile_rank out of range");
        build_tile_list(c, a.w, a.h, a.rank, a.ranks);
        if (!c->tile_count && !c->tile_host.empty()) {
            CU(c, c->tiles.reserve(c->tile_host.size() * 4));
            CU(c, cudaMemcpyAsync(c->tiles.p, c->tile_host.data(), c->tile_host.size() * 4, cudaMemcpyHostToDevice, st));
            CU(c, cudaStreamSynchronize(st));
            c->tile_count = (uint32_t)c->tile_host.size();
        }
        W.n_macro_x = (a.w + kMacroTile - 1) / kMacroTile;
        units_all = c->tile_host.size();
    } else {
        if (a.n == 0 || a.k >= a.n) return fail(c, LGB_ERR_INVALID, "capture_subset: need k < n");
        W.sub_n = a.n;
        units_all = area > a.k ? (area - a.k + a.n - 1) / a.n : 0;
        W.compact_out = 1;
    }
    const uint64_t px_per_unit = a.mode == 0 ? (uint64_t)kMacroTile * kMacroTile : 1;
    set_divisors(W, s->cam.root);
    set_camera_constants(W, s->cam);
    const uint64_t total_all = units_all * px_per_unit * W.spp;
    if (s->cam.pixel_separation != 0.0 && W.aspect > 4.0)
        return fail(c, LGB_ERR_UNSUPPORTED, "orthographic capture with aspect > 4: the scene's coordinate bound assumed aspect <= 4");
    const DevScene& S = s->dev;
    const uint32_t nl = std::max<uint32_t>(S.n_lights, 1);
    // automatic: where a bundle of >= 8 rays shares a traversal that is long enough to be worth sharing (measured: a loss on
    // scenes of a few dozen primitives, a gain on large ones)
    W.beams = (W.spp >= 4 && !S.instanced && (c->beams == 1 || (c->beams < 0 && W.spp >= 8 && large_scene(S)))) ? 1u : 0u;
    if (!a.klog_no_camgrid && total_all) if (int rc = ensure_camgrid(c, s, a.w, a.h, total_all, W, st)) return rc;
    if (!S.nodes && total_all && (!W.cg_start || !(S.grids && !S.instanced) || S.general)) {
        // a scene created without its BVH (lgb_scene::Deferred) meets a frame that walks one: build it now, then the grids again
        if (int rc = ensure_bvh(c, s)) return rc;
        W.cg_start = nullptr; W.cg_entries = nullptr; W.cg_large = nullptr;
        W.beams = (W.spp >= 4 && !S.instanced && (c->beams == 1 || (c->beams < 0 && W.spp >= 8 && large_scene(S)))) ? 1u : 0u;
        if (!a.klog_no_camgrid) if (int rc = ensure_camgrid(c, s, a.w, a.h, total_all, W, st)) return rc;
    }
    const bool grid_shadows = S.grids && !S.instanced;                 // no shadow queues, no occluder cache
    // hit setup inside the camera-grid kernel (no k_setup launch): plain captures whose shadows go through the light grids
    W.setup_in_primary = (c->setup_in_primary && W.cg_start && grid_shadows && !a.aov && a.mode != 3) ? 1u : 0u;
    const bool beam_lists = W.beams && (!W.cg_start || !grid_shadows); // pixel beams (primary) and / or shadow beams
    const bool two_lists = beam_lists && !grid_shadows && S.n_lights > 1 && c->side_streams && c->side.n;
    const bool need_radiance = !render_fused(W.spp) || S.general || a.want_li;
    const bool lazy_ties = s->lazy_fn && !s->dev.rank;
    // the queue area also lends its first words to the pixel beams' fallback list and to k_shade's list of specular slots (one u32 per slot)
    const uint32_t queue_nl = grid_shadows ? ((beam_lists || S.specular) ? 1u : 0u) : nl;
    // ---- how much of the frame one band may hold
    uint64_t per_slot = 8 + 24 + 4 + 4 + 4 + 1 + 12 * (uint64_t)queue_nl + (need_radiance ? 24 : 0);
    if (S.specular && S.recursion > 0 && c->whitted_wavefront) per_slot += sizeof(SpawnRec) + 2 * 48 + 24 + 8 + 24 + 4 + 4 + 4 + 1;      // level buffers, worst case per slot
    const uint64_t per_pixel = (grid_shadows ? 0 : 4 * (uint64_t)nl) + (beam_lists ? (uint64_t)kBeamList * 8 + 8 : 0) + (two_lists ? (uint64_t)kBeamList * 8 + 4 : 0);
    const uint64_t unit_bytes = px_per_unit * (per_pixel + per_slot * W.spp), unit_slots = px_per_unit * W.spp;
    uint64_t units_band = std::max<uint64_t>(1, std::min<uint64_t>(c->wave_budget / std::max<uint64_t>(unit_bytes, 1), ((1ull << 32) - 65) / unit_slots));
    if (unit_slots >= (1ull << 32) - 64) return fail(c, LGB_ERR_INVALID, "capture: more than 2^32 samples in one macro tile");
    units_band = std::min<uint64_t>(units_band, std::max<uint64_t>(units_all, 1));
    const uint64_t n_bands = units_all ? (units_all + units_band - 1) / units_band : 0;
    const uint64_t slots_band = std::max<uint64_t>(units_band * unit_slots, 1), npix_band = std::max<uint64_t>(units_band * px_per_unit, 1);
    if (need_radiance) CU(c, c->radiance.reserve(slots_band * 3 * sizeof(double)));
    CU(c, c->counters.reserve(kCtrBytes));
    CU(c, c->wave.reserve(wave_bytes(slots_band, queue_nl, grid_shadows ? 0 : npix_band)));
    char* const wave_base = (char*)c->wave.p;
    CU(c, c->wave_ctr.reserve(kWaveCtrBytes));
    if (beam_lists) CU(c, c->beam.reserve(npix_band * kBeamList * sizeof(uint2) + npix_band * 8));
    if (two_lists) CU(c, c->beam2.reserve(npix_band * kBeamList * sizeof(uint2) + npix_band * 4));
    if (lazy_ties) CU(c, c->ties.reserve((size_t)kTieCap * 4));
    DevOut O{};
    O.radiance = (double*)c->radiance.p;
    O.counters = (DevCounters*)c->counters.p;
    if (a.d_film) O.film = (uint8_t*)a.d_film;
    else {
        CU(c, c->film.reserve(std::max<uint64_t>(a.mode == 0 ? area : units_all, 1) * 4));
        O.film = (uint8_t*)c->film.p;
    }
    if (a.aov) {
        CU(c, c->aov_id.reserve(area * W.spp * 4)); CU(c, c->aov_t.reserve(area * W.spp * 8)); CU(c, c->aov_occl.reserve(area * W.spp * 4));
        O.aov_id = (uint32_t*)c->aov_id.p; O.aov_t = (double*)c->aov_t.p; O.aov_occl = (uint32_t*)c->aov_occl.p;
        if (a.want_li) { CU(c, c->aov_li.reserve(std::max<uint64_t>(area * W.spp, 1) * 24)); O.aov_li = (double*)c->aov_li.p; }
    }
    CU(c, cudaMemsetAsync(c->counters.p, 0, kCtrBytes, st));
    CU(c, cudaEventRecord(c->ev0, st));
    cudaEvent_t* pev = (stats && sync_stats && total_all) ? c->phase : nullptr;
    uint32_t tie_slots = 0;
    const bool st_on = a.aov || c->count_work;
    const SideStreams* side = (c->side_streams && c->side.n && !a.klog) ? &c->side : nullptr;
    uint64_t level_rays = 0; uint32_t level_launches = 0;
    float phase_ms[6] = {0, 0, 0, 0, 0, 0};
    int wf = 0;
    // lgb_capture of a whole frame on one device, one band: the shade kernel runs in slices and the film's finished rows leave for the
    // host behind each (the read-back of a 33 MB film costs 1.7 ms behind the frame, 0.5 ms behind its last slice)
    c->host_film_done = false;
    ShadeChunks chunk_rec{}; ShadeChunks* chunks = nullptr;
    constexpr uint32_t kShadeSlices = 4;
    if (a.host_film && a.mode == 0 && a.ranks == 1 && n_bands == 1 && !a.aov && !a.klog && !a.d_film && !S.general && area * 4 >= (8u << 20) && !std::getenv("LGB_NO_FILM_OVERLAP")) {
        if (!c->copy_stream) CU(c, cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
        CU(c, c->reserve_chunk_events(2 * kShadeSlices));
        chunk_rec.want = kShadeSlices; chunk_rec.ev = c->chunk_ev.data();
        chunks = &chunk_rec;
    }
    for (uint64_t band = 0; band < n_bands; band++) {
        const uint64_t u0 = band * units_band, un = std::min<uint64_t>(units_band, units_all - u0);
        if (a.mode == 0) {
            W.tile_list = (const uint32_t*)c->tiles.p + u0; W.n_tiles = (uint32_t)un;
            W.n_pixels = un * px_per_unit;
        } else {
            W.sub_k = (uint64_t)a.k + u0 * (uint64_t)a.n; W.compact_base = u0;
            W.n_pixels = un;
        }
        const uint64_t total = W.n_pixels * W.spp;
        DevWave V = carve_wave(wave_base, c->wave_ctr.p, slots_band, queue_nl, grid_shadows ? 0 : npix_band);
        if (beam_lists) {
            V.beam_list = (uint2*)c->beam.p; V.beam_count = (uint32_t*)((char*)c->beam.p + npix_band * kBeamList * sizeof(uint2));
            V.beam_bound = (float*)(V.beam_count + npix_band);
            if (two_lists) { V.beam_list2 = (uint2*)c->beam2.p; V.beam_count2 = (uint32_t*)((char*)c->beam2.p + npix_band * kBeamList * sizeof(uint2)); }
        }
        V.tie_list = nullptr; V.tie_cap = 0;
        if (s->lazy_fn && !s->dev.rank) {
            V.tie_list = (uint32_t*)c->ties.p; V.tie_cap = kTieCap;
            if (const char* e = std::getenv("LGB_TIE_CAP")) V.tie_cap = std::min<uint32_t>(kTieCap, (uint32_t)std::strtoul(e, nullptr, 10));   // tests: force the whole-frame re-trace
        }
        wf = (S.general && c->whitted_wavefront) ? 4 : 0;               // launch_render stops after k_shade; the levels and the resolve follow here
        if (wf && S.specular && S.recursion > 0 && total) {             // k_shade of the camera wave spawns level 1
            CU(c, c->lvl_ctr.reserve(4 * (kMaxRecursion + 2) * 4));
            CU(c, cudaMemsetAsync(c->lvl_ctr.p, 0, 4 * (kMaxRecursion + 2) * 4, st));
            if (!prepare_spawn(c, V, 0, total)) wf = 0;                 // not enough memory for the level buffers: one thread per ray tree instead
        }
        if (s->lazy_fn && !s->dev.rank && total) {
            // no rank tables yet: trace the primary rays, and only if one met two primitives at bit-identical t fetch the
            // caller's reference tree, build the tables and re-trace those slots (lasgun_b200.h, "Lazy reference tree")
            if (int rc = sync_scene_copy(c, s, st)) return rc;
            CU(c, launch_render(S, s->cam, s->shade, W, O, V, st_on, a.aov, c->sm_count, st, pev, 1, side, a.klog));
            uint32_t ties = 0;
            CU(c, cudaMemcpyAsync(&ties, V.tie_count, 4, cudaMemcpyDeviceToHost, st));
            CU(c, cudaStreamSynchronize(st));
            if (ties) {
                if (int rc = ensure_rank_tables(c, s)) return rc;
                s->tie_retraces += ties; tie_slots += ties;
                if (!S.nodes && s->deferred.scratch) {
                    // the re-trace walks the BVH, and this scene was created without one (lgb_scene::Deferred): build it -- that re-orders
                    // the primitives, so the hits of this band are void -- and render the band again, now with resident rank tables
                    if (c->leader) return fail(c, LGB_ERR_INVALID, "internal: a device-group replica met an exact-t tie without a BVH");
                    if (int rc = ensure_bvh(c, s)) return rc;
                    W.cg_start = nullptr; W.cg_entries = nullptr; W.cg_large = nullptr;
                    if (!a.klog_no_camgrid) if (int rc = ensure_camgrid(c, s, a.w, a.h, total_all, W, st)) return rc;
                    band--;                                      // (unsigned wrap at band 0 is undone by the loop's increment)
                    continue;
                }
                W.setup_in_primary = 0;                          // the re-traced slots change their hits: k_setup runs over the band after all
                DevWork W2 = W;
                DevCounters before{};
                if (ties <= V.tie_cap) { W2.slot_list = V.tie_list; W2.n_list = ties; }
                else if (band == 0) CU(c, cudaMemsetAsync(c->counters.p, 0, kCtrBytes, st));          // too many to list: the whole band again
                (void)before;
                if (int rc = sync_scene_copy(c, s, st)) return rc;
                CU(c, launch_render(s->dev, s->cam, s->shade, W2, O, V, st_on, a.aov, c->sm_count, st, ties <= V.tie_cap ? nullptr : pev, 1, side, a.klog));
            }
            if (int rc = sync_scene_copy(c, s, st)) return rc;
            CU(c, launch_render(s->dev, s->cam, s->shade, W, O, V, st_on, a.aov, c->sm_count, st, pev, 2 | wf, side, a.klog, chunks));
        } else {
            if (int rc = sync_scene_copy(c, s, st)) return rc;
            CU(c, launch_render(s->dev, s->cam, s->shade, W, O, V, st_on, a.aov, c->sm_count, st, pev, 3 | wf, side, a.klog, chunks));
        }
        if (wf && total) {                     // materials beyond plastic: the levels of the specular ray trees, then the film
            if (S.specular && S.recursion > 0) if (int rc = run_whitted_levels(c, s, O, total, st, stats != nullptr, &level_rays, &level_launches)) return rc;
            if (pev) CU(c, cudaEventRecord(pev[5], st));
            CU(c, launch_resolve(W, O, st));
            if (pev) CU(c, cudaEventRecord(pev[6], st));
        }
        if (O.aov_li) CU(c, launch_export_li(W, O, V, st));
        if (pev && n_bands > 1) {              // the phase events are re-recorded by the next band: read them now
            CU(c, cudaStreamSynchronize(st));
            for (int k = 0; k < 6; k++) { float pm = 0.f; CU(c, cudaEventElapsedTime(&pm, c->phase[k], c->phase[k + 1])); phase_ms[k] += pm; }
        }
    }
    CU(c, cudaEventRecord(c->ev1, st));
    if (!s->last_use) CU(c, cudaEventCreateWithFlags(&s->last_use, cudaEventDisableTiming));
    CU(c, cudaEventRecord(s->last_use, st));
    uint32_t copy_rows[9] = {0};                 // film rows [copy_rows[k], copy_rows[k + 1]) leave behind slice k
    bool copy_bounce = false;
    if (chunks && chunks->launched) {
        cudaPointerAttributes at{};
        if (cudaPointerGetAttributes(&at, a.host_film) != cudaSuccess) { cudaGetLastError(); copy_bounce = true; }
        else copy_bounce = at.type == cudaMemoryTypeUnregistered;
        if (copy_bounce) CU(c, c->reserve_film_host(area * 4));
        char* dst = copy_bounce ? (char*)c->film_host : (char*)a.host_film;
        const uint64_t px_tile_row = (uint64_t)W.n_macro_x * kMacroTile * kMacroTile;
        for (uint32_t k = 0; k < chunks->launched; k++) {
            const uint64_t rows = k + 1 == chunks->launched ? a.h : std::min<uint64_t>(a.h, chunks->done_pixels[k] / px_tile_row * kMacroTile);
            copy_rows[k + 1] = (uint32_t)std::max<uint64_t>(rows, copy_rows[k]);
            CU(c, cudaStreamWaitEvent(c->copy_stream, chunks->ev[k], 0));
            const size_t off = (size_t)copy_rows[k] * a.w * 4, len = (size_t)(copy_rows[k + 1] - copy_rows[k]) * a.w * 4;
            if (len) CU(c, cudaMemcpyAsync(dst + off, (const char*)O.film + off, len, cudaMemcpyDeviceToHost, c->copy_stream));
            CU(c, cudaEventRecord(chunks->ev[kShadeSlices + k], c->copy_stream));
        }
        CU(c, cudaEventRecord(c->ev2, c->copy_stream));
    }
    if (stats && sync_stats) {
        DevCounters hc;
        CU(c, launch_fold_counters((DevCounters*)c->counters.p, st));
        CU(c, cudaMemcpyAsync(&hc, c->counters.p, sizeof hc, cudaMemcpyDeviceToHost, st));
        CU(c, cudaStreamSynchronize(st));
        std::memset(stats, 0, sizeof *stats);
        stats->primary_rays = hc.primary_rays; stats->primary_hits = hc.primary_hits;
        stats->shadow_rays = hc.primary_hits * s->dev.n_lights;
        stats->shadow_rays_traced = hc.shadow_traced; stats->shadow_occluded = hc.shadow_occluded; stats->shadow_cache_hits = hc.shadow_cached;
        stats->node_tests = hc.node_tests; stats->primary_node_tests = hc.p_node_tests;
        for (int k = 0; k < 3; k++) { stats->primary_filter_tests[k] = hc.p_filter[k]; stats->primary_exact_tests[k] = hc.p_exact[k]; }
        if (total_all && n_bands == 1) for (int k = 0; k < 6; k++) { float pm = 0.f; CU(c, cudaEventElapsedTime(&pm, c->phase[k], c->phase[k + 1])); stats->kernel_ms[k] = pm; }
        else for (int k = 0; k < 6; k++) stats->kernel_ms[k] = phase_ms[k];
        for (int k = 0; k < 3; k++) { stats->filter_tests[k] = hc.filter[k]; stats->exact_tests[k] = hc.exact[k]; }
        stats->stack_overflow = hc.stack_overflow;
        stats->beams = W.beams; stats->tie_retraces = tie_slots; stats->secondary_rays = hc.secondary_rays + level_rays;
        const bool one_kernel = surface_fused(S, W, O, a.aov);              // k_surface: setup + shadows + shade + film
        const uint32_t shadow_launches = grid_shadows ? 1u                                                                // k_gshadow
                                         : s->dev.n_lights * (W.spp > 1 ? 3 : 1) + ((W.beams && W.spp > 1 && !S.instanced) ? 2 * s->dev.n_lights : 0);      // + k_sbeam + k_swalk per light
        const uint32_t primary_launches = W.cg_start ? 1u : (W.beams && W.spp >= 4 && !S.instanced) ? 3u : 1u;           // k_cprimary | k_beam + k_leafp + fallback | k_primary
        const uint32_t shade_launches = S.general ? (S.specular && S.recursion && !wf ? 3u : 2u) : (render_fused(W.spp) && !O.aov_li) ? 1u : 2u;
        const uint32_t setup_launches = (W.setup_in_primary || setup_fused(S, W, O, a.aov)) ? 0u : 1u;                                          // (inside k_gshadow otherwise)
        stats->kernel_launches = total_all ? level_launches + (uint32_t)n_bands * (primary_launches + (one_kernel ? 1u : setup_launches + shadow_launches + shade_launches)) : 0;
        if (chunks && chunks->launched) stats->kernel_launches += chunks->launched - 1;
        stats->bands = (uint32_t)n_bands;
        float ms = 0.f; CU(c, cudaEventElapsedTime(&ms, c->ev0, c->ev1));
        stats->render_ms = ms; stats->total_ms = ms;
    }
    if (chunks && chunks->launched) {
        for (uint32_t k = 0; k < chunks->launched; k++) {
            CU(c, cudaEventSynchronize(chunks->ev[kShadeSlices + k]));
            const size_t off = (size_t)copy_rows[k] * a.w * 4, len = (size_t)(copy_rows[k + 1] - copy_rows[k]) * a.w * 4;
            if (copy_bounce && len) {
                const char* src = (const char*)c->film_host + off; char* out = (char*)a.host_film + off;
                Pool::get().for_range(len, 256u << 10, [&](size_t b, size_t e, size_t) { std::memcpy(out + b, src + b, e - b); });
            }
        }
        CU(c, cudaStreamSynchronize(st));           // (the slices' events are behind everything on st but the counters' copy)
        if (stats && sync_stats) { float ms = 0.f; CU(c, cudaEventElapsedTime(&ms, c->ev0, c->ev2)); stats->total_ms = ms; }
        c->host_film_done = true;
    }
    return LGB_OK;
}

// capture over a device group (lib.rs:55-104: one blocking call, every worker): device k of n renders the macro tiles of rank k
// into the leader's film -- the peers' uchar4 stores cross NVLink while their other tiles are still being shaded, no collective
// and no gather pass -- each on its own host thread (a capture holds short synchronisation points: tile-list upload, the
// lazy-tree tie count, the statistics), and the call returns when every device's stream is drained.
static int group_capture(lgb_ctx* c, lgb_scene* s, uint32_t w, uint32_t h, void* film, lgb_stats* stats) {
    const uint32_t n = 1 + (uint32_t)c->peers.size();
    if (s->replicas.size() != c->peers.size()) return fail(c, LGB_ERR_INVALID, "capture: the scene was not created on this device group");
    if (!s->dev.nodes && s->deferred.scratch) {          // deferred BVH: the leader decides for the group before anybody renders
        CU(c, cudaSetDevice(c->device));
        DevWork Wp{};
        const uint64_t samples = (uint64_t)w * h * s->cam.root * s->cam.root;
        if (int rc = ensure_camgrid(c, s, w, h, samples, Wp, c->stream)) return rc;
        if (!Wp.cg_start || !(s->dev.grids && !s->dev.instanced) || s->dev.general) if (int rc = ensure_bvh(c, s)) return rc;
    }
    std::vector<int> rc(n, LGB_OK);
    std::vector<lgb_stats> st(n);
    std::vector<std::thread> workers;
    for (uint32_t k = 1; k < n; k++)
        workers.emplace_back([&, k] {
            CaptureArgs a{w, h, 0, k, n, 0, 0, false, film, nullptr};
            rc[k] = run_capture(c->peers[k - 1], s->replicas[k - 1], a, &st[k], true);
        });
    {
        CaptureArgs a{w, h, 0, 0, n, 0, 0, false, film, nullptr};
        rc[0] = run_capture(c, s, a, &st[0], true);
    }
    for (std::thread& t : workers) t.join();
    cudaSetDevice(c->device);
    for (uint32_t k = 1; k < n; k++) if (rc[k]) return fail(c, rc[k], "device " + std::to_string(c->peers[k - 1]->device) + ": " + c->peers[k - 1]->error);
    if (rc[0]) return rc[0];
    if (stats) {
        *stats = st[0];
        for (uint32_t k = 1; k < n; k++) {
            const lgb_stats& o = st[k];
            stats->primary_rays += o.primary_rays; stats->primary_hits += o.primary_hits; stats->shadow_rays += o.shadow_rays;
            stats->shadow_rays_traced += o.shadow_rays_traced; stats->shadow_occluded += o.shadow_occluded; stats->shadow_cache_hits += o.shadow_cache_hits;
            stats->node_tests += o.node_tests; stats->primary_node_tests += o.primary_node_tests; stats->secondary_rays += o.secondary_rays;
            for (int t = 0; t < 3; t++) {
                stats->exact_tests[t] += o.exact_tests[t]; stats->filter_tests[t] += o.filter_tests[t];
                stats->primary_exact_tests[t] += o.primary_exact_tests[t]; stats->primary_filter_tests[t] += o.primary_filter_tests[t];
            }
            for (int t = 0; t < 6; t++) stats->kernel_ms[t] = std::max(stats->kernel_ms[t], o.kernel_ms[t]);
            stats->render_ms = std::max(stats->render_ms, o.render_ms); stats->total_ms = std::max(stats->total_ms, o.total_ms);
            stats->kernel_launches += o.kernel_launches; stats->stack_overflow |= o.stack_overflow; stats->tie_retraces += o.tie_retraces;
        }
    }
    return LGB_OK;
}

int lgb_capture_device(lgb_ctx* c, lgb_scene* s, uint32_t w, uint32_t h, uint32_t rank, uint32_t ranks, void* d_film, void* stream, lgb_stats* stats) {
    if (!d_film) return fail(c, LGB_ERR_INVALID, "lgb_capture_device: d_film is NULL");
    if (c && !c->peers.empty() && ranks == 1) {              // device group: the whole frame, split over the group; blocking
        if (stream) CU(c, cudaStreamSynchronize((cudaStream_t)stream));        // the caller's earlier work on the film (a clear) is done
        lgb_stats local;
        return group_capture(c, s, w, h, d_film, stats ? stats : &local);
    }
    CaptureArgs a{w, h, 0, rank, ranks, 0, 0, false, d_film, (cudaStream_t)stream};
    return run_capture(c, s, a, stats, stats != nullptr);
}

// The film goes to the caller's buffer.  A pageable one (the reference's Film is a Vec, film.rs:22-45) makes cudaMemcpy bounce through
// the driver's own small pinned buffers at ~13 GB/s; instead the film crosses PCIe in chunks into a pinned buffer of the context's at
// the link's rate, and every host thread carries a chunk on into the caller's memory while the next one is crossing.
static int finish_host(lgb_ctx* c, const void* dev, void* host, size_t bytes, lgb_stats* stats) {
    constexpr size_t kChunk = 4u << 20;
    bool bounce = bytes >= 2 * kChunk && !std::getenv("LGB_NO_FILM_BOUNCE");
    if (bounce) {
        cudaPointerAttributes at{};
        if (cudaPointerGetAttributes(&at, host) != cudaSuccess) { cudaGetLastError(); bounce = false; }
        else bounce = at.type == cudaMemoryTypeUnregistered;
    }
    if (bounce && c->reserve_film_host(bytes) != cudaSuccess) { cudaGetLastError(); bounce = false; }
    if (bounce) {
        const size_t n = (bytes + kChunk - 1) / kChunk;
        CU(c, c->reserve_chunk_events(n));
        for (size_t i = 0; i < n; i++) {
            const size_t off = i * kChunk, len = std::min(kChunk, bytes - off);
            CU(c, cudaMemcpyAsync((char*)c->film_host + off, (const char*)dev + off, len, cudaMemcpyDeviceToHost, c->stream));
            CU(c, cudaEventRecord(c->chunk_ev[i], c->stream));
        }
        CU(c, cudaEventRecord(c->ev2, c->stream));
        for (size_t i = 0; i < n; i++) {
            const size_t off = i * kChunk, len = std::min(kChunk, bytes - off);
            CU(c, cudaEventSynchronize(c->chunk_ev[i]));
            const char* src = (const char*)c->film_host + off; char* dst = (char*)host + off;
            Pool::get().for_range(len, 256u << 10, [&](size_t b, size_t e, size_t) { std::memcpy(dst + b, src + b, e - b); });
        }
        if (stats) { float ms = 0.f; CU(c, cudaEventElapsedTime(&ms, c->ev0, c->ev2)); stats->total_ms = ms; }
        return LGB_OK;
    }
    CU(c, cudaMemcpyAsync(host, dev, bytes, cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaEventRecord(c->ev2, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    if (stats) { float ms = 0.f; CU(c, cudaEventElapsedTime(&ms, c->ev0, c->ev2)); stats->total_ms = ms; }
    return LGB_OK;
}

int lgb_capture(lgb_ctx* c, lgb_scene* s, uint32_t w, uint32_t h, uint8_t* rgba, lgb_stats* stats) {
    if (!rgba) return fail(c, LGB_ERR_INVALID, "lgb_capture: rgba_out is NULL");
    lgb_stats local; lgb_stats* stp = stats ? stats : &local;
    int rc;
    if (c && !c->peers.empty()) {
        if (w == 0 || h == 0 || (uint64_t)w * h >= (1ull << 32)) return fail(c, LGB_ERR_INVALID, "capture: bad film size");
        CU(c, cudaSetDevice(c->device));
        CU(c, c->film.reserve((size_t)w * h * 4));
        CU(c, cudaEventRecord(c->ev0, c->stream));
        rc = group_capture(c, s, w, h, c->film.p, stp);
    } else {
        CaptureArgs a{w, h, 0, 0, 1, 0, 0, false, nullptr, nullptr};
        a.host_film = rgba;
        rc = run_capture(c, s, a, stp, true);
    }
    if (rc) return rc;
    if (stp->stack_overflow) return fail(c, LGB_ERR_UNSUPPORTED, "traversal stack overflow");
    if (c->peers.empty() && c->host_film_done) return LGB_OK;         // the film left in slices behind the shade kernel's (run_capture)
    return finish_host(c, c->film.p, rgba, (size_t)w * h * 4, stp);
}

int lgb_capture_aov(lgb_ctx* c, lgb_scene* s, uint32_t w, uint32_t h, uint8_t* rgba, uint32_t* prim_id, double* t, uint32_t* occl, double* li, lgb_stats* stats) {
    lgb_stats local; lgb_stats* stp = stats ? stats : &local;
    CaptureArgs a{w, h, 0, 0, 1, 0, 0, true, nullptr, nullptr};
    a.want_li = li != nullptr;
    int rc = run_capture(c, s, a, stp, true);
    if (rc) return rc;
    const uint64_t ns = (uint64_t)w * h * s->cam.root * s->cam.root;
    if (prim_id) CU(c, cudaMemcpyAsync(prim_id, c->aov_id.p, ns * 4, cudaMemcpyDeviceToHost, c->stream));
    if (t) CU(c, cudaMemcpyAsync(t, c->aov_t.p, ns * 8, cudaMemcpyDeviceToHost, c->stream));
    if (occl) CU(c, cudaMemcpyAsync(occl, c->aov_occl.p, ns * 4, cudaMemcpyDeviceToHost, c->stream));
    if (li) CU(c, cudaMemcpyAsync(li, c->aov_li.p, ns * 24, cudaMemcpyDeviceToHost, c->stream));
    if (rgba) return finish_host(c, c->film.p, rgba, (size_t)w * h * 4, stp);
    CU(c, cudaStreamSynchronize(c->stream));
    return LGB_OK;
}

int lgb_capture_subset(lgb_ctx* c, lgb_scene* s, uint32_t k, uint32_t n, uint32_t w, uint32_t h, uint8_t* rgba, lgb_stats* stats) {
    if (!rgba) return fail(c, LGB_ERR_INVALID, "lgb_capture_subset: rgba_inout is NULL");
    lgb_stats local; lgb_stats* stp = stats ? stats : &local;
    CaptureArgs a{w, h, 1, 0, 1, k, n, false, nullptr, nullptr};
    int rc = run_capture(c, s, a, stp, true);
    if (rc) return rc;
    const uint64_t area = (uint64_t)w * h;
    const uint64_t np = area > k ? (area - k + n - 1) / n : 0;
    std::vector<uint8_t> compact(np * 4);
    if (np) { rc = finish_host(c, c->film.p, compact.data(), np * 4, stp); if (rc) return rc; }
    for (uint64_t p = 0; p < np; p++) std::memcpy(rgba + (k + p * (uint64_t)n) * 4, &compact[4 * p], 4);   // lib.rs:152-161
    return LGB_OK;
}

int lgb_capture_profile(lgb_ctx* c, lgb_scene* s, uint32_t w, uint32_t h, void* d_film, lgb_kernel_time* out, uint32_t cap, uint32_t* n_out, lgb_stats* stats) {
    if (!c || !out || !n_out) return fail(c, LGB_ERR_INVALID, "lgb_capture_profile: NULL argument");
    CU(c, cudaSetDevice(c->device));
    CU(c, c->klog_snaps.reserve(sizeof(DevCounters) * KernelLog::kMax));
    c->klog.n = 0; c->klog.snaps = (DevCounters*)c->klog_snaps.p;
    lgb_stats local; lgb_stats* stp = stats ? stats : &local;
    CaptureArgs a{w, h, 0, 0, 1, 0, 0, false, d_film, nullptr};
    a.klog = &c->klog;
    if (int rc = run_capture(c, s, a, stp, true)) return rc;             // synchronises
    const int n = c->klog.n;
    std::vector<DevCounters> snap((size_t)std::max(n, 1));
    if (n) CU(c, cudaMemcpy(snap.data(), c->klog.snaps, sizeof(DevCounters) * n, cudaMemcpyDeviceToHost));
    DevCounters prev{};
    for (int i = 0; i < n && (uint32_t)i < cap; i++) {
        lgb_kernel_time& o = out[i];
        std::memset(&o, 0, sizeof o);
        std::snprintf(o.name, sizeof o.name, "%s", c->klog.name[i]);
        CU(c, cudaEventElapsedTime(&o.ms, c->klog.ev0[i], c->klog.ev1[i]));
        const DevCounters& k = snap[i];
        o.node_tests = k.node_tests - prev.node_tests;
        for (int t = 0; t < 3; t++) { o.filter_tests[t] = k.filter[t] - prev.filter[t]; o.exact_tests[t] = k.exact[t] - prev.exact[t]; }
        o.primary_rays = k.primary_rays - prev.primary_rays; o.primary_hits = k.primary_hits - prev.primary_hits;
        o.shadow_rays = k.shadow_traced - prev.shadow_traced; o.shadow_occluded = k.shadow_occluded - prev.shadow_occluded;
        prev = k;
    }
    *n_out = (uint32_t)n;
    return LGB_OK;
}

int lgb_trace_rays(lgb_ctx* c, lgb_scene* s, const double* rays, uint64_t n, uint32_t* ids, double* ts, double* ng, double* ns) {
    if (!c || !s || (!rays && n)) return fail(c, LGB_ERR_INVALID, "lgb_trace_rays: NULL argument");
    // The f32 error bound of the traversal is derived from the box of the scene and its camera (lgb_scene::origin_lo/hi).  k_trace
    // starts the f32 ray of an origin outside it where the ray enters the box grown by 1/64 of its extent.  Origins farther out
    // than one extent E of the box are refused: there the reference's own f64 tests lose so much to cancellation (a sphere's
    // |o - c|^2 - r^2) that their hits stray from the surface by more than the conservative culls allow for.
    TraceBox B;
    double M = 0.0, E = 0.0;
    for (int k = 0; k < 3; k++) {
        M = std::max(M, std::max(std::fabs(s->origin_lo[k]), std::fabs(s->origin_hi[k])));
        E = std::max(E, s->origin_hi[k] - s->origin_lo[k]);
    }
    E += M * std::ldexp(1.0, -10);
    for (int k = 0; k < 3; k++) { B.lo[k] = s->origin_lo[k] - E / 64.0; B.hi[k] = s->origin_hi[k] + E / 64.0; }
    for (uint64_t i = 0; i < n; i++) {
        const double* o = rays + 6 * i;
        for (int k = 0; k < 3; k++) {
            if (o[k] >= s->origin_lo[k] - E && o[k] <= s->origin_hi[k] + E) continue;
            char msg[400];
            std::snprintf(msg, sizeof msg, "lgb_trace_rays: the origin (%.17g, %.17g, %.17g) of ray %llu lies more than %.17g (one extent) outside the box "
                          "[%.17g, %.17g] x [%.17g, %.17g] x [%.17g, %.17g] of the scene and its camera", o[0], o[1], o[2], (unsigned long long)i, E,
                          s->origin_lo[0], s->origin_hi[0], s->origin_lo[1], s->origin_hi[1], s->origin_lo[2], s->origin_hi[2]);
            return fail(c, LGB_ERR_UNSUPPORTED, msg);
        }
    }
    CU(c, cudaSetDevice(c->device));
    if (int rc = ensure_bvh(c, s)) return rc;
    if (n == 0) return LGB_OK;
    const size_t need = n * (48 + 4 + 8 + 24 + 24);
    CU(c, c->scratch.reserve(need));
    char* base = (char*)c->scratch.p;
    double* d_rays = (double*)base; double* d_t = (double*)(base + n * 48); double* d_ng = (double*)(base + n * 56); double* d_ns = (double*)(base + n * 80);
    uint32_t* d_id = (uint32_t*)(base + n * 104);
    CU(c, cudaMemcpyAsync(d_rays, rays, n * 48, cudaMemcpyHostToDevice, c->stream));
    if (int rc = sync_scene_copy(c, s, c->stream)) return rc;
    CU(c, launch_trace(s->dev, B, d_rays, n, d_id, d_t, d_ng, d_ns, c->stream));
    if (ids) CU(c, cudaMemcpyAsync(ids, d_id, n * 4, cudaMemcpyDeviceToHost, c->stream));
    if (ts) CU(c, cudaMemcpyAsync(ts, d_t, n * 8, cudaMemcpyDeviceToHost, c->stream));
    if (ng) CU(c, cudaMemcpyAsync(ng, d_ng, n * 24, cudaMemcpyDeviceToHost, c->stream));
    if (ns) CU(c, cudaMemcpyAsync(ns, d_ns, n * 24, cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    return LGB_OK;
}

int lgb_debug_fastmath(lgb_ctx* c, const double* x, uint64_t n, double* rcp_out, double* rsqrt_out) {
    if (!c || (n && (!x || !rcp_out || !rsqrt_out))) return fail(c, LGB_ERR_INVALID, "lgb_debug_fastmath: NULL argument");
    CU(c, cudaSetDevice(c->device));
    if (n == 0) return LGB_OK;
    CU(c, c->scratch.reserve(n * 24));
    double* d = (double*)c->scratch.p;
    CU(c, cudaMemcpyAsync(d, x, n * 8, cudaMemcpyHostToDevice, c->stream));
    CU(c, launch_fastmath(d, n, d + n, d + 2 * n, c->stream));
    CU(c, cudaMemcpyAsync(rcp_out, d + n, n * 8, cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaMemcpyAsync(rsqrt_out, d + 2 * n, n * 8, cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    return LGB_OK;
}

// ---------------------------------------------------------------------------------------- ceilings
int lgb_measure_l2_read_gbs(lgb_ctx* c, uint64_t bytes, int iters, double* out) {
    if (!c || !out || bytes < 4096 || iters < 1) return fail(c, LGB_ERR_INVALID, "lgb_measure_l2_read_gbs: bad argument");
    CU(c, cudaSetDevice(c->device));
    bytes &= ~(uint64_t)15;
    CU(c, c->scratch.reserve(bytes + 16));
    CU(c, cudaMemsetAsync(c->scratch.p, 0, bytes + 16, c->stream));
    float* sink = (float*)((char*)c->scratch.p + bytes);
    CU(c, launch_l2_read(c->scratch.p, bytes, 2, sink, c->sm_count, c->stream));   // warm L2
    CU(c, cudaEventRecord(c->ev0, c->stream));
    CU(c, launch_l2_read(c->scratch.p, bytes, iters, sink, c->sm_count, c->stream));
    CU(c, cudaEventRecord(c->ev1, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    float ms = 0.f; CU(c, cudaEventElapsedTime(&ms, c->ev0, c->ev1));
    *out = (double)bytes * iters / (ms * 1e-3) / 1e9;
    return LGB_OK;
}
int lgb_measure_fp32_gops(lgb_ctx* c, int iters, double* out) {
    if (!c || !out || iters < 1) return fail(c, LGB_ERR_INVALID, "lgb_measure_fp32_gops: bad argument");
    CU(c, cudaSetDevice(c->device));
    CU(c, c->scratch.reserve(64));
    CU(c, launch_fp32_peak(iters / 8 + 1, (float*)c->scratch.p, c->sm_count, c->stream));
    CU(c, cudaEventRecord(c->ev0, c->stream));
    CU(c, launch_fp32_peak(iters, (float*)c->scratch.p, c->sm_count, c->stream));
    CU(c, cudaEventRecord(c->ev1, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    float ms = 0.f; CU(c, cudaEventElapsedTime(&ms, c->ev0, c->ev1));
    *out = (double)c->sm_count * 8 * 256 * 8.0 * iters / (ms * 1e-3) / 1e9;    // FFMA lane-instructions per second (GHz-lanes)
    return LGB_OK;
}
int lgb_measure_fp64_gops(lgb_ctx* c, int iters, double* out) {
    if (!c || !out || iters < 1) return fail(c, LGB_ERR_INVALID, "lgb_measure_fp64_gops: bad argument");
    CU(c, cudaSetDevice(c->device));
    CU(c, c->scratch.reserve(64));
    CU(c, launch_fp64_peak(iters / 8 + 1, (double*)c->scratch.p, c->sm_count, c->stream));
    CU(c, cudaEventRecord(c->ev0, c->stream));
    CU(c, launch_fp64_peak(iters, (double*)c->scratch.p, c->sm_count, c->stream));
    CU(c, cudaEventRecord(c->ev1, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    float ms = 0.f; CU(c, cudaEventElapsedTime(&ms, c->ev0, c->ev1));
    *out = (double)c->sm_count * 8 * 256 * 8.0 * iters / (ms * 1e-3) / 1e9;
    return LGB_OK;
}

}  // extern "C"
