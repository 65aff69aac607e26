// Device-side scene layout shared by the kernels and the C-ABI glue (lgb_api.cu).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/lasgun_b200.h"

namespace lgb {

constexpr int kStackDepth = 64;          // bvh.rs:469 — the reference's fixed traversal stack
constexpr int kMacroTile = 32;           // macro tile edge in pixels (multi-GPU interleave unit)
constexpr int kMicroW = 8, kMicroH = 4;  // one warp of pixels at 1 spp
constexpr uint32_t kNoNormals = 0xFFFFFFFFu;
#ifndef LGB_LEAF_CONSTANTS
#define LGB_LEAF_CONSTANTS
constexpr uint32_t kLeafBit = 0x80000000u;       // child word encoding, see lgb_build.hpp
constexpr uint32_t kLeafFirstMask = 0x00FFFFFFu;
#endif
constexpr uint32_t kDone = 0x7FFFFFFFu;          // traversal sentinel (never a valid node index)
constexpr int kMaxSpaceDepth = 8;                // nested transformed aggregates along one path
constexpr uint32_t kSpaceIdentity = 1u, kSpaceSwap = 2u;
constexpr uint32_t kNoParent = 0xFFFFFFFFu;

// World box of the scene and its camera (lgb_scene::origin_lo/hi) grown by a margin: k_trace starts the f32 ray of a caller-supplied
// ray whose origin lies outside it where the ray enters it.
struct TraceBox { double lo[3], hi[3]; };

// One coordinate system of the scene (lgb_build.hpp): cgmath column-major Transform3 of the aggregate that opens it.
struct DevSpace {
    double m[16], minv[16];
    uint32_t parent, depth, root_node, flags;
    float err_abs; uint32_t pad[3];
};

// Light grid (lgb_grid.cu): cube map around a point light, 6 faces x res^2 cells; cell (face, v, u) lists the primitives whose
// direction footprint seen from the light touches it as (type << 30 | index, lower bound of the distance from the light as float
// bits), nearest first; `large`: the primitives with footprints of more than kGridLargeCells cells, tested by every ray.
constexpr uint32_t kGridSortMax = 0xFFFFFFFFu;   // every cell's list is sorted nearest first (cub::DeviceSegmentedSort, lgb_grid.cu)
struct DevGrid {
    const uint32_t* cell_start;   // 6 res^2 + 1
    const uint2* entries;
    const uint2* large;
    uint32_t res, n_large;
    double map[6][4];             // per face {u0, su, v0, sv}: direction (u, v) lies in cell (floor((u - u0) su), floor((v - v0) sv)), clamped to the
                                  // face's res x res cells -- the cells are laid over the part of the face the scene's small primitives cover
};

// All pointers are device pointers.  Layout (see DESIGN.md §3):
//   nodes      4 x float4 per node: child0 {lo.xyz, hi.xyz}, child1 {lo.xyz, hi.xyz}, {child0, child1, -, -};
//              boxes padded (conservative for f32 rays); child word = node index, or
//              kLeafBit | type << 29 | (count - 1) << 24 | first  (homogeneous leaf, primitives stored in leaf order)
//   sph32      float4 {c.xyz, r} f32 copy for the filter; sph64 4 doubles exact (same index)
//   cub32      2 x float4 padded {lo, hi}; cub64 6 doubles exact
//   tri        3 x float4 {p0, id} {p1, material} {p2, normals_index|kNoNormals}
//   tri_nrm    9 floats per entry (indexed by the value stored in tri[3i+2].w)
//   rank       8 x prim_count u32: reference traversal position per direction octant (exact-t ties only)
//   materials  kMatStride doubles {c0.xyz, p0, c1.xyz, flags, p1, p2, -, -}: the record of include/lasgun_b200.h (c0 = kd | eta | kr,
//              c1 = ks | k | kt, p0 = roughness | sigma | u_roughness | eta) with flags = bit0 diffuse lobe, bit1 glossy lobe,
//              bit2 a material the plastic fast path does not evaluate (Oren-Nayar, metal, glass, mirror), bit3 specular lobes
//              (glass, mirror: Whitted recursion), kind << 8; p1 = v_roughness (metal) | Oren-Nayar A, p2 = Oren-Nayar B
//   lights     9 doubles {pos, intensity, falloff}
struct DevScene {
    const float4* nodes;
    const float4* sph32;
    const double* sph64;
    const uint32_t* sph_mat;
    const uint32_t* sph_id;
    const float4* cub32;
    const double* cub64;
    const uint32_t* cub_mat;
    const uint32_t* cub_id;
    const float4* tri;
    const float* tri_nrm;
    const uint32_t* rank;
    const double* materials;
    const double* lights;
    const DevSpace* spaces;       // instanced scenes only (n_spaces > 1 or a transformed root)
    const uint32_t* inst_space;   // leaf-ordered child-space ids (leaf type LGB_PRIM_INSTANCE)
    const uint32_t* sph_space; const uint32_t* cub_space; const uint32_t* tri_space;   // space of every primitive, leaf order
    const DevGrid* grids;         // one per light, or NULL: shadow rays traverse the BVH (instanced or small scenes)
    uint32_t n_sph, n_cub, n_tri; // primitives per type (the leaf-ordered arrays above)
    uint32_t prim_count;
    uint32_t rank_items;          // prim_count + n_spaces: stride of one octant's rank table
    uint32_t n_spaces;
    uint32_t instanced;
    uint32_t n_lights;
    uint32_t n_nodes;
    uint32_t general;     // some material carries flag bit2: the GENERAL shade variant runs
    uint32_t specular;    // some material carries flag bit3: k_secondary follows the specular rays
    uint32_t recursion;   // scene.recursion (scene.rs:60), depth limit of integrate.rs:69
    float err_abs;        // absolute coordinate error bound of an f32 ray against this scene (see lgb_api.cu)
    // This record once more, in global memory (uploaded before every launch sequence, lgb_api.cu): what an out-of-line device function
    // reads.  A `const DevScene&` bound to the kernel's parameter block has its address taken, and then every thread copies the whole
    // record to its stack at entry (28 STL.64) whether or not it ever makes the call.
    const DevScene* self;
};

struct DevCamera {
    double origin[3], view[3], up[3], aux[3];
    double image_plane_height, pixel_separation, sample_distance;
    uint32_t root;
};

struct DevShade {
    double ambient[3];
    double bg_inner[3], bg_outer[3], bg_scale;
};

// Which pixels a launch renders.
//   mode 0: macro tiles listed in tile_list (tile index = my * n_macro_x + mx)
//   mode 1: capture_subset — pixels k, k+n, ... of the row-major film (lib.rs:152)
//   mode 2: caller-supplied rays (lgb_trace_rays)
//   mode 3: one level of the specular ray trees (Whitted recursion): slot i is ray i of `rays`, spp = 1
struct DevWork {
    uint32_t mode;
    uint32_t w, h;
    double winv, hinv, aspect;       // film.rs:36-45
    const uint32_t* tile_list;
    uint32_t n_tiles;
    uint32_t n_macro_x;
    uint64_t sub_k; uint32_t sub_n;  // (sub_k: k plus the pixels of the bands before this one)
    uint64_t compact_base;           // mode 1: film index of this band's first pixel
    uint64_t n_pixels;               // pixel slots in this launch
    uint32_t spp;
    // the per-launch constants of camera.rs:115-118,131-133, formed once on the host with the reference's own operations (IEEE doubles,
    // no contraction: the same bits every thread would compute): ipw = iph * aspect, updiff = up * sep, auxdiff = aux * sep,
    // halfdiff = updiff * 0.5 + auxdiff * 0.5 with sep = sample_distance * (iph * hinv)
    double cam_ipw, cam_updiff[3], cam_auxdiff[3], cam_halfdiff[3];
    uint64_t fd_spp, fd_root, fd_nmx; // ceil(2^64 / d) for d = spp, the supersampling root, n_macro_x (0: d == 1): fdiv(), lgb_kernels.cu
    uint32_t anchor;                 // sample index of the pixel's anchor shadow ray (centre of the sample grid)
    const uint32_t* slot_list;       // k_primary: trace only these sample slots (re-trace of unresolved exact-t ties) ...
    uint64_t n_list;                 // ... this many of them ...
    const uint32_t* n_list_dev;      // ... or as many as this device counter says (beam fallback)
    uint32_t compact_out;            // resolve writes film[slot] instead of film[y*w + x]
    uint32_t beams;                  // primary rays through pixel beams (k_beam / k_leafp) when spp >= 4
    // camera grid (lgb_grid.cu): the primary rays of a perspective camera walk the primitive list of their pixel tile (k_cprimary)
    const uint32_t* cg_start;        // NULL: no camera grid for this launch
    const uint2* cg_entries;
    const uint2* cg_large;
    uint32_t cg_n_large, cg_shift, cg_nx;
    uint32_t setup_in_primary;       // k_cprimary<SETUP> does k_setup's work (plain captures with light grids; run_capture decides)
    const double* rays;              // mode 3: origin + direction, 6 doubles per slot
    uint32_t depth;                  // mode 3: depth of these rays in integrate.rs:23's recursion (camera rays: 0)
    uint32_t hole_lo, hole_hi;       // mode 3: slots [hole_lo, hole_hi) hold no ray (reflected rays fill the level's slots from 0, transmitted ones from hole_hi)
    uint32_t block_off;              // k_shade_lean<FUSED> launched in chunks (ShadeChunks): blockIdx.x + block_off is the block's place in the whole launch
};


// One specular hit and the rays it spawned (k_spawn); k_gather folds the children's radiance back into the parent's:
// output + reflected + refracted, integrate.rs:79, with reflected = spectrum x li (:103) and refracted = spectrum x li * |wi.ns| / pdf (:129)
struct SpawnRec {
    uint32_t slot;                   // the parent's slot in its own level
    uint32_t child_r, child_t;       // ray indices in the next level, or kNoChild
    uint32_t pad;
    double spec_r[3], spec_t[3], c;  // c = |wi . ns| of the transmitted direction (pdf = 1)
};
constexpr uint32_t kNoChild = 0xFFFFFFFFu;

struct DevCounters {
    unsigned long long primary_rays, primary_hits, shadow_traced, shadow_occluded, shadow_cached;
    unsigned long long node_tests;     // node fetches (each tests two child boxes)
    unsigned long long filter[3];    // f32 filter tests by primitive type (sphere, cuboid, triangle)
    unsigned long long exact[3];     // f64 reference-arithmetic tests by primitive type
    unsigned long long p_node_tests, p_filter[3], p_exact[3];   // the share of the primary-ray kernels in the three counters above
    unsigned long long beam_node_tests;                         // of those: node fetches of the pixel beams (k_beam)
    unsigned long long secondary_rays;                          // rays k_secondary traced
    unsigned int stack_overflow;
    unsigned int pad;
};

// Where the kernels add: the buffer behind DevOut::counters holds the record the host reads, then kCtrStripes copies kCtrStride bytes
// apart; a warp adds to the copy its block and warp index select (ctr(), lgb_kernels.cu) and launch_fold_counters sums the copies into
// the record before anybody reads it.  With ONE copy the 4 M warps of k_cprimary sent 8 M atomics to two words per frame; the L2 slice
// those words lived on was the kernel's bottleneck whenever a hot read-only line of the frame (tile list, large list, lights) happened
// to share it -- 6.8 ms or 8.2-8.8 ms for the same launch, decided by whatever the process had allocated before (profiles/r2_v36-38).
constexpr uint32_t kCtrStripes = 512, kCtrStride = 256;       // (64 stripes still cost 0.2 ms per grid walk: 130 k atomics per line)
static_assert(sizeof(DevCounters) <= kCtrStride, "counter stripe");
constexpr size_t kCtrBytes = (size_t)(1 + kCtrStripes) * kCtrStride;
cudaError_t launch_fold_counters(DevCounters* base, cudaStream_t stream);

// lgb_capture_profile: CUDA events around every kernel launch of one frame (all on ONE stream for that call, so a launch's
// duration is its own) and a snapshot of the work counters behind each, so that every launch's share of them is known.  Host-side only.
struct KernelLog {
    static constexpr int kMax = 64;
    char name[kMax][40];
    cudaEvent_t ev0[kMax], ev1[kMax];
    int n = 0, made = 0;
    DevCounters* snaps = nullptr;        // device, kMax entries: the counters as they stand after launch i
    void begin(const char* nm, int light, cudaStream_t s) {
        if (n >= kMax) return;
        if (n >= made) { cudaEventCreate(&ev0[n]); cudaEventCreate(&ev1[n]); made = n + 1; }
        if (light >= 0) snprintf(name[n], sizeof name[n], "%s[light %d]", nm, light); else snprintf(name[n], sizeof name[n], "%s", nm);
        cudaEventRecord(ev0[n], s);
    }
    void end(cudaStream_t s, const DevCounters* ctr) {
        if (n >= kMax) return;
        cudaEventRecord(ev1[n], s);
        if (snaps && ctr) { launch_fold_counters(const_cast<DevCounters*>(ctr), s); cudaMemcpyAsync(snaps + n, ctr, sizeof(DevCounters), cudaMemcpyDeviceToDevice, s); }
        n++;
    }
};

// The fused shade + film kernel launched as `want` consecutive slices, an event behind each: lgb_capture starts the film's trip to
// the host behind the first slice instead of behind the frame (launch_render fills launched / done_pixels; host-side only).
struct ShadeChunks { uint32_t want; cudaEvent_t* ev; uint32_t launched; uint64_t done_pixels[8]; };
// Side streams for the per-light shadow chains (launch_render); host-side only.
struct SideStreams { cudaStream_t s[3]; cudaEvent_t fork, join[3]; int n; };

// Wavefront buffers, one entry per sample slot g = pixel_slot * spp + s.
struct DevWave {
    double* hit_t;                   // closest-hit parameter (f64, reference arithmetic)
    uint32_t* hit_ref;               // type << 30 | index, LGB_MISS, or kSlotUnused (pixel outside the film)
    double* ps;                      // shadow-ray origin p + p_err (3 per slot)
    uint32_t* occl;                  // bit l set: light l occluded
    uint32_t* gate;                  // bit l set: wi of light l and wo lie on the same side of ng (bsdf.rs:75,85-86); k_setup -> k_shade (lean path)
    unsigned char* sflags;           // the reference's sign decisions about the surface record (kSf*, lgb_kernels.cu); k_setup -> k_shade
    // Shadow-ray queues of slot indices, three per light (kQueueA/B/C), each queue_stride entries:
    //   A  anchor rays: the centre sample of every pixel (every ray at 1 spp); traced first, their occluder
    //      is remembered per (light, pixel) in `occluder`
    //   B  the other samples of the pixel: k_pretest runs the exact test of the remembered occluder alone
    //   C  the B rays that the remembered occluder does not block: full any-hit traversal
    uint32_t* queue;                 // [(light * 3 + which) * queue_stride + i]
    uint64_t queue_stride;
    uint32_t* occluder;              // [light * n_pixels + pixel_slot]: ref of the anchor ray's occluder or LGB_MISS
    unsigned long long* work_counter;   // [0] primary fetch counter; then u32 queue_count[lights][3], queue_fetch[lights][3]
    uint32_t* queue_count;
    uint32_t* queue_fetch;
    uint32_t* tie_count;             // exact-t ties k_primary could not resolve (scene without resident rank tables)
    uint32_t* tie_list;              // their sample slots (first tie_cap of them)
    uint32_t tie_cap;
    // pixel beams (k_beam / k_leafp): leaves reached by the bundle of a pixel's sample rays, nearest first
    uint2* beam_list;                // [i * n_pixels + pixel_slot] = (leaf word, entry distance bits)
    uint32_t* beam_count;            // per pixel slot; kBeamOverflow: fall back to the per-ray traversal
    float* beam_bound;               // per pixel slot: the list is complete for rays whose closest hit is not beyond it
    uint32_t* free_count;            // per light: anchor rays k_shadow found free, listed (in that light's still empty queue C) for k_sbeam
    uint2* beam_list2;               // the same pair once more: shadow beams of the light whose chain runs on the side stream
    uint32_t* beam_count2;
    uint32_t* fallback_list;         // sample slots of such pixels (aliases the shadow queues, which are not yet in use)
    uint32_t* fallback_count;
    uint32_t* sec_list;              // sample slots whose closest hit has specular lobes (aliases the shadow queues, drained by then)
    uint32_t* sec_count;
    // wavefront Whitted recursion: k_shade turns the specular hits of this wave into the rays of the next level
    SpawnRec* recs;                  // NULL: list the slots in sec_list instead (k_secondary follows)
    double* next_rays;               // 6 doubles per ray of the next level
    uint32_t* spawn_ctr;             // {records written, reflected rays, transmitted rays, -}
    uint32_t next_t_base;            // first slot of the transmitted rays in the next level (= slots of this wave)
};
constexpr int kQueueA = 0, kQueueB = 1, kQueueC = 2;
constexpr size_t kWaveCtrBytes = 8 + 4 * (size_t)LGB_MAX_LIGHTS * 3 * 2 + 16 + 4 * (size_t)LGB_MAX_LIGHTS;     // + tie_count, fallback_count, sec_count, pad, free_count[lights]
constexpr int kMatStride = 12;
constexpr uint32_t kMatDiffuse = 1u, kMatGlossy = 2u, kMatGeneral = 4u, kMatSpecular = 8u;
constexpr uint32_t kMaxRecursion = 12;         // depth of the per-ray stack k_secondary keeps (lgb_scene_create rejects deeper scenes)
constexpr uint32_t kTieCap = 1u << 20;
#ifndef LGB_BEAM_LIST
#define LGB_BEAM_LIST 24             // entries a bundle may list before the pixel goes the per-ray way; 16 / 24 / 32 / 48 / 64: 44.4 / 44.6 / 44.7 / 45.1 / 45.2 ms/frame on mixed4k
#endif
constexpr int kBeamList = LGB_BEAM_LIST;                  // leaves a pixel beam may reach before the pixel falls back to per-ray traversal
constexpr uint32_t kBeamOverflow = 0xFFFFFFFFu;
constexpr uint32_t kEntryDone = 0xFFFFFFFFu;       // a queue-B entry k_swalk has resolved from the pixel's shadow beam
constexpr uint32_t kSlotUnused = 0xFFFFFFFEu;

struct DevOut {
    double* radiance;                // 3 doubles per sample slot (slot = pixel_slot * spp + s)
    uint32_t* aov_id;                // optional, global sample index
    double* aov_t;
    uint32_t* aov_occl;
    double* aov_li;                  // optional: the radiance of every sample (li, integrate.rs:23), global sample index
    DevCounters* counters;           // optional
    uint8_t* film;                   // row-major RGBA8, or the (h, w, 3) f32 linear film of lgb_capture_linear (may be a peer pointer)
};

// lgb_capture_guides: per-pixel geometry of the camera rays' closest hits (k_guides), row-major; NULL outputs are not written.
struct DevGuides {
    float* normal;                   // (h, w, 3): in-order sum of the samples' shading normals times 1/spp
    float* depth;                    // (h, w): t of the anchor sample times |view|, +inf on a miss
    uint32_t* prim_id;               // (h, w): canonical id of the anchor sample's hit, or LGB_MISS
    float* coverage;                 // (h, w): samples that hit / spp
    double view_len;                 // |view| (host, f64)
};

}  // namespace lgb
