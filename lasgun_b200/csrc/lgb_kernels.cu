// Render kernels: camera rays -> closest-hit traversal -> plastic shading with point-light shadow
// rays -> per-sample radiance; resolve -> RGBA8 film.  sm_100a, compiled with -fmad=false.
//
// Precision scheme (DESIGN.md §4): traversal culling and primitive *filters* run in f32 and are
// conservative (they never reject what the reference's f64 test would accept); every candidate
// that survives is re-tested with the reference's own f64 arithmetic (lgb_math.cuh), so the
// closest-hit primitive and its t are the reference's, and shading runs in f64 in the
// reference's operation order (integrate.rs:23-80).
#include <math_constants.h>

#include <algorithm>

#include "lgb_math.cuh"

namespace lgb {

// Wavefront entries (6 GB per mixed4k frame, each written once and read once) are stored / loaded with the streaming hint
// (st.global.cs / ld.global.cs: evict-first in L2), so they do not push the scene and the grids (~100-160 MB) out of the 126 MB L2.
template <class T> __device__ __forceinline__ void wst(T* p, T v) { __stcs(p, v); }
template <class T> __device__ __forceinline__ T wld(const T* p) { return __ldcs(p); }

// ------------------------------------------------------------------ per-ray f32 state
struct RayF {
    float ox, oy, oz;
    float ix, iy, iz;        // 1/d, clamped to +-1e30 (rounded from the f64 reciprocal)
    float nx, ny, nz;        // -o * (1/d): slab planes are evaluated as fma(plane, 1/d, -o/d)
    float dx, dy, dz;
    float inv_dd, inv_len;   // 1/(d.d), 1/|d|
    float sx, sy, sz;        // triangle shear (triangle.rs:199-201), f32 copies
    float err;               // absolute coordinate error bound; +inf disables the filters
    int kz;
    unsigned oct;            // bit a set <=> dir_is_neg[a] (bvh.rs:463)
};

__device__ __forceinline__ float clamp_idir(float d) {
    const float v = 1.0f / d;                  // <= 1 ulp from the exact reciprocal: inside the 2^-20 slack of the node test
    return fabsf(v) > 1e30f ? copysignf(1e30f, v) : v;
}

// The f32 ray starts at `o` (a point of the line of r): r.o itself, or for caller-supplied rays from far away the point where the
// line enters the scene's box (k_trace).  The f64 exact tests always see r.
__device__ __forceinline__ RayF make_rayf_at(const Ray64& r, const D3 o, float err_abs) {
    RayF f;
    f.ox = (float)o.x; f.oy = (float)o.y; f.oz = (float)o.z;
    f.dx = (float)r.d.x; f.dy = (float)r.d.y; f.dz = (float)r.d.z;
    // dir_is_neg[a] = (1 / d[a] < 0) (bvh.rs:463, ray.rs:28-33) is the sign bit of d[a], -0 included: no f64 division needed
    f.oct = (signbit(r.d.x) ? 1u : 0u) | (signbit(r.d.y) ? 2u : 0u) | (signbit(r.d.z) ? 4u : 0u);
    f.ix = clamp_idir(f.dx); f.iy = clamp_idir(f.dy); f.iz = clamp_idir(f.dz);
    f.nx = -f.ox * f.ix; f.ny = -f.oy * f.iy; f.nz = -f.oz * f.iz;
    float dd = f.dx * f.dx + f.dy * f.dy + f.dz * f.dz;
    f.inv_dd = 1.0f / dd;
    f.inv_len = rsqrtf(dd);
    // |d| outside the comfortable f32 range: make every filter band infinite (exact tests only).
    f.err = (dd > 1e-24f && dd < 1e24f) ? err_abs : CUDART_INF_F;
    f.kz = max_dimension_abs(r.d);
    const int kx = (f.kz + 1) % 3, ky = (kx + 1) % 3;
    float fdz = f.kz == 0 ? f.dx : (f.kz == 1 ? f.dy : f.dz);
    float fdx = kx == 0 ? f.dx : (kx == 1 ? f.dy : f.dz);
    float fdy = ky == 0 ? f.dx : (ky == 1 ? f.dy : f.dz);
    f.sz = 1.0f / fdz;
    f.sx = -fdx * f.sz;
    f.sy = -fdy * f.sz;
    return f;
}
__device__ __forceinline__ RayF make_rayf(const Ray64& r, float err_abs) { return make_rayf_at(r, r.o, err_abs); }
// The f32 ray of r advanced to parameter t0 >= 0 (k_trace).  Its t values are those of r minus t0: every cull that compares them
// with the best hit only gets weaker, and nothing the scene holds lies before t0 (t0 is the entry into a box around the scene).
__device__ __forceinline__ RayF make_rayf(const Ray64& r, float err_abs, double t0) {
    return make_rayf_at(r, d3(r.o.x + t0 * r.d.x, r.o.y + t0 * r.d.y, r.o.z + t0 * r.d.z), err_abs);
}

// Conservative slab test of an f32 ray against a padded f32 box (DESIGN.md §4.1): returns false only if the
// exact f64 ray certainly misses the exact box or enters it beyond the best hit.  Every computed t carries a
// relative error <= ~3 ulp, so the interval test widens tfar by (1 + 2^-20) and the caller passes
// tbest_up = best * (1 + 2^-20); the sign of tfar is exact.  tnear (raw) orders the children.
__device__ __forceinline__ bool slab2(float lx, float ly, float lz, float hx, float hy, float hz, const RayF& f, float tbest_up, float& tnear_out) {
    float t1x = __fmaf_rn(lx, f.ix, f.nx), t2x = __fmaf_rn(hx, f.ix, f.nx);
    float t1y = __fmaf_rn(ly, f.iy, f.ny), t2y = __fmaf_rn(hy, f.iy, f.ny);
    float t1z = __fmaf_rn(lz, f.iz, f.nz), t2z = __fmaf_rn(hz, f.iz, f.nz);
    float tnear = fmaxf(fmaxf(fminf(t1x, t2x), fminf(t1y, t2y)), fminf(t1z, t2z));
    float tfar = fminf(fminf(fmaxf(t1x, t2x), fmaxf(t1y, t2y)), fmaxf(t1z, t2z));
    tnear_out = tnear;
    return tnear <= tfar * (1.0f + 9.5367431640625e-7f) && tfar > 0.0f && tnear <= tbest_up;
}
// Same test specialised on the ray's direction octant (bit a of OCT set <=> d[a] < 0): the near / far plane of
// every axis is known at compile time, so the six min/max that order t1, t2 disappear, and the `tfar > 0` and
// best-hit tests fold into one compare: max(tnear, 0) <= min(tfar (1 + 2^-20), tbest_up).  It accepts
// whatever slab2 accepts (plus tfar == 0, which is merely conservative).
template <int OCT>
__device__ __forceinline__ bool slab_oct(float lx, float ly, float lz, float hx, float hy, float hz, const RayF& f, float tbest_up, float& tnear_out) {
    const float tnx = __fmaf_rn((OCT & 1) ? hx : lx, f.ix, f.nx), tfx = __fmaf_rn((OCT & 1) ? lx : hx, f.ix, f.nx);
    const float tny = __fmaf_rn((OCT & 2) ? hy : ly, f.iy, f.ny), tfy = __fmaf_rn((OCT & 2) ? ly : hy, f.iy, f.ny);
    const float tnz = __fmaf_rn((OCT & 4) ? hz : lz, f.iz, f.nz), tfz = __fmaf_rn((OCT & 4) ? lz : hz, f.iz, f.nz);
    const float tnear = fmaxf(fmaxf(tnx, tny), tnz);
    const float tfar = fminf(fminf(tfx, tfy), tfz) * (1.0f + 9.5367431640625e-7f);
    tnear_out = tnear;
    return fmaxf(tnear, 0.0f) <= fminf(tfar, tbest_up);
}
__device__ __forceinline__ float inflate_up(double t) { return __double2float_ru(t) * (1.0f + 9.5367431640625e-7f); }

struct Hit { double t; uint32_t ref; };     // ref = type << 30 | index in the leaf-ordered arrays

// the counter stripe of this warp (lgb_types.cuh, kCtrStripes)
__device__ __forceinline__ DevCounters* ctr(const DevOut& O) {
    return reinterpret_cast<DevCounters*>(reinterpret_cast<char*>(O.counters) + (size_t)(1u + ((blockIdx.x + (threadIdx.x >> 5) * 17u) & (kCtrStripes - 1u))) * kCtrStride);
}
struct LocalCounters { unsigned int node_tests, filter[3], exact[3]; };

__device__ __forceinline__ uint32_t canonical_id(const DevScene& S, uint32_t ref) {
    const uint32_t type = ref >> 30, idx = ref & 0x3FFFFFFFu;
    if (type == LGB_PRIM_SPHERE) return S.sph_id[idx];
    if (type == LGB_PRIM_CUBOID) return S.cub_id[idx];
    return __float_as_uint(S.tri[3 * (size_t)idx].w);
}

// ------------------------------------------------------------------ spaces (nested transformed aggregates)
// Transform3::inverse_transform_ray (transform.rs:279-283) with cgmath's Matrix4 * Vector4 = c0 x + c1 y + c2 z + c3 w
// (w = 1 for the origin, 0 for the direction; the matrices are affine, so transform_point's division by w is by 1).
__device__ __forceinline__ D3 m4_apply(const double* m, D3 v, double w) {
    return d3(m[0] * v.x + m[4] * v.y + m[8] * v.z + m[12] * w,
              m[1] * v.x + m[5] * v.y + m[9] * v.z + m[13] * w,
              m[2] * v.x + m[6] * v.y + m[10] * v.z + m[14] * w);
}
__device__ __forceinline__ Ray64 ray_into(const DevSpace& sp, const Ray64& r) {
    Ray64 o; o.o = m4_apply(sp.minv, r.o, 1.0); o.d = m4_apply(sp.minv, r.d, 0.0);
    return o;
}
// The world ray taken down the chain of transforms to `space`, level by level as the reference does (bvh.rs:462).
// (Out of line, so it takes the space table by value: see DevScene::self.)
__device__ __noinline__ Ray64 ray_to_space(const DevSpace* spaces, uint32_t space, const Ray64& world) {
    uint32_t chain[kMaxSpaceDepth]; int n = 0;
    for (uint32_t s = space; s != kNoParent; s = spaces[s].parent) chain[n++] = s;
    Ray64 r = world;
    while (n--) { const DevSpace& sp = spaces[chain[n]]; if (!(sp.flags & kSpaceIdentity)) r = ray_into(sp, r); }
    return r;
}
__device__ __forceinline__ Ray64 ray_to_space(const DevScene& S, uint32_t space, const Ray64& world) { return ray_to_space(S.spaces, space, world); }
__device__ __forceinline__ uint32_t space_of(const DevScene& S, uint32_t ref) {
    const uint32_t type = ref >> 30, idx = ref & 0x3FFFFFFFu;
    return type == LGB_PRIM_SPHERE ? S.sph_space[idx] : type == LGB_PRIM_CUBOID ? S.cub_space[idx] : S.tri_space[idx];
}
__device__ __forceinline__ unsigned octant_of(const Ray64& r) {                  // bvh.rs:463 on Ray::new's dinv (ray.rs:28-33)
    return (1.0 / r.d.x < 0.0 ? 1u : 0u) | (1.0 / r.d.y < 0.0 ? 2u : 0u) | (1.0 / r.d.z < 0.0 ? 4u : 0u);
}
// Exact-t tie between two primitives of an instanced scene: both are lifted to their deepest common space (a nested
// level stands for everything below it) and compared by that level's test order for the ray's octant THERE.
__device__ __noinline__ bool rank_before_instanced(const DevScene* Sg, const Ray64& world, uint32_t ref_a, uint32_t ref_b) {
    const DevScene& S = *Sg;              // the record in global memory (DevScene::self)
    uint32_t ia = canonical_id(S, ref_a), sa = space_of(S, ref_a), ib = canonical_id(S, ref_b), sb = space_of(S, ref_b);
    uint32_t da = S.spaces[sa].depth, db = S.spaces[sb].depth;
    while (da > db) { ia = S.prim_count + sa; sa = S.spaces[sa].parent; da--; }
    while (db > da) { ib = S.prim_count + sb; sb = S.spaces[sb].parent; db--; }
    while (sa != sb) { ia = S.prim_count + sa; sa = S.spaces[sa].parent; ib = S.prim_count + sb; sb = S.spaces[sb].parent; }
    const Ray64 r = ray_to_space(S, sa, world);
    const uint32_t* rk = S.rank + (size_t)octant_of(r) * S.rank_items;
    return rk[ia] < rk[ib];
}

// A candidate with exact parameter t replaces the current best iff it is nearer, or equally near and
// earlier in the reference's own traversal order for this ray's octant (lgb_build.hpp).
// Without resident rank tables (lazy reference tree, lgb_api.cu) the tie is only RECORDED: the caller re-traces the ray
// once the tables exist.
template <bool INST>
__device__ __forceinline__ bool accepts(const DevScene& S, const RayF& f, const Ray64& world, const Hit& best, double t, uint32_t ref, uint32_t& tied) {
    if (t < best.t) return true;
    if (t == best.t && best.ref != LGB_MISS && best.ref != ref) {
        if (!S.rank) { tied = 1u; return false; }
        if (INST) return rank_before_instanced(S.self, world, ref, best.ref);
        const uint32_t* r = S.rank + (size_t)f.oct * S.rank_items;
        return r[canonical_id(S, ref)] < r[canonical_id(S, best.ref)];
    }
    return false;
}

// f32 filter for one triangle, specialised on the ray's dominant axis (no per-vertex selects).
template <int KZ>
__device__ __forceinline__ bool tri_filter(const float4 q0, const float4 q1, const float4 q2, const RayF& f, float best_tf) {
    constexpr int KX = (KZ + 1) % 3, KY = (KX + 1) % 3;
    const float o[3] = {f.ox, f.oy, f.oz};
    const float a[3] = {q0.x - o[0], q0.y - o[1], q0.z - o[2]};
    const float b[3] = {q1.x - o[0], q1.y - o[1], q1.z - o[2]};
    const float c[3] = {q2.x - o[0], q2.y - o[1], q2.z - o[2]};
    const float Ax = __fmaf_rn(f.sx, a[KZ], a[KX]), Ay = __fmaf_rn(f.sy, a[KZ], a[KY]);
    const float Bx = __fmaf_rn(f.sx, b[KZ], b[KX]), By = __fmaf_rn(f.sy, b[KZ], b[KY]);
    const float Cx = __fmaf_rn(f.sx, c[KZ], c[KX]), Cy = __fmaf_rn(f.sy, c[KZ], c[KY]);
    const float e0 = __fmaf_rn(Bx, Cy, -By * Cx), e1 = __fmaf_rn(Cx, Ay, -Cy * Ax), e2 = __fmaf_rn(Ax, By, -Ay * Bx);
    const float m = fmaxf(fmaxf(fmaxf(fabsf(Ax), fabsf(Ay)), fmaxf(fabsf(Bx), fabsf(By))), fmaxf(fabsf(Cx), fabsf(Cy)));
    const float band = 6.0f * m * f.err;
    const float emin = fminf(fminf(e0, e1), e2), emax = fmaxf(fmaxf(e0, e1), e2);
    if (emin < -band && emax > band) return false;
    // depth range of the triangle along the ray
    const float tz0 = a[KZ] * f.sz, tz1 = b[KZ] * f.sz, tz2 = c[KZ] * f.sz;
    const float tlo = fminf(fminf(tz0, tz1), tz2), thi = fmaxf(fmaxf(tz0, tz1), tz2);
    const float slack = f.err * fabsf(f.sz);
    if (tlo - slack - fabsf(tlo) * 1e-6f > best_tf) return false;
    if (thi + slack + fabsf(thi) * 1e-6f < 0.0f) return false;
    return true;
}

// Closest hit (ANYHIT = false) or "any hit with t < tmax" (ANYHIT = true, shadow rays: the reference
// asks for the closest t and compares it with 1.0, light/point.rs:48-49, which is equivalent).
// while-while traversal of the device BVH: the inner loop descends interior nodes (two child boxes per
// fetch, nearer child first), the outer loop intersects one homogeneous leaf.  The `tnear > best` cull is
// result-safe because every primitive rejects t >= isect.t itself (bvh.rs:473 never looks at isect.t).
struct Trav {                 // resumable traversal state of one ray
    Hit best;
    float best_tf, best_up;
    uint32_t cur;
    int sp;
    uint32_t space;           // instanced scenes: the space the ray is in right now
    uint32_t tied;            // an exact-t tie could not be resolved (no rank tables resident)
    __device__ __forceinline__ void init(double tmax, uint32_t root = 0) {
        best.t = tmax; best.ref = LGB_MISS; best_tf = __double2float_ru(tmax); best_up = inflate_up(tmax); cur = root; sp = 0; space = 0; tied = 0;
    }
};

// Inner loop of the while-while traversal: descend interior nodes until `cur` is a leaf or kDone.
// OCT < 8: every ray of the warp has that direction octant (slab_oct); OCT == 8: mixed warp (slab2).
// TSTACK (closest-hit rays): the entry distance of a deferred child is kept beside it, and a popped entry
// that now starts beyond the best hit is dropped without fetching its node.
template <bool TSTACK>
__device__ __forceinline__ uint32_t stack_pop(int& sp, const uint32_t* stack, const float* tstack, float best_up) {
    while (sp) {
        --sp;
        if (!TSTACK || tstack[sp] <= best_up) return stack[sp];
    }
    return kDone;
}
template <int OCT, bool STATS, bool TSTACK>
__device__ __forceinline__ void node_loop(const DevScene& S, const RayF& f, float best_up, uint32_t& cur, int& sp, uint32_t* stack, float* tstack, LocalCounters& lc) {
    while (!(cur & kLeafBit) && cur != kDone) {
        const float4* np = S.nodes + 4 * (size_t)cur;
        const float4 n0 = __ldg(np), n1 = __ldg(np + 1), n2 = __ldg(np + 2);
        const float2 n3 = __ldg(reinterpret_cast<const float2*>(np + 3));
        if (STATS) lc.node_tests++;
        float tn0, tn1;
        bool h0, h1;
        if (OCT < 8) {
            h0 = slab_oct<OCT & 7>(n0.x, n0.y, n0.z, n0.w, n1.x, n1.y, f, best_up, tn0);
            h1 = slab_oct<OCT & 7>(n1.z, n1.w, n2.x, n2.y, n2.z, n2.w, f, best_up, tn1);
        } else {
            h0 = slab2(n0.x, n0.y, n0.z, n0.w, n1.x, n1.y, f, best_up, tn0);
            h1 = slab2(n1.z, n1.w, n2.x, n2.y, n2.z, n2.w, f, best_up, tn1);
        }
        const uint32_t c0 = __float_as_uint(n3.x), c1 = __float_as_uint(n3.y);
        if (h0 && h1) {
            const bool swap = tn1 < tn0;
            cur = swap ? c1 : c0;
            if (TSTACK) tstack[sp] = swap ? tn0 : tn1;
            stack[sp] = swap ? c0 : c1; sp++;
        } else if (h0) cur = c0;
        else if (h1) cur = c1;
        else cur = stack_pop<TSTACK>(sp, stack, tstack, best_up);
    }
}

// The primitives of one leaf against one ray: conservative f32 filter, then the reference's exact f64 test
// (DESIGN.md 4).  ANYHIT: returns true as soon as one is hit with t < tmax (T.best holds it); otherwise T.best is
// updated and the result is false.
template <bool ANYHIT, bool STATS, bool INST>
__device__ __forceinline__ bool leaf_prims(const DevScene& S, const Ray64& world, const Ray64& ray, const RayF& f, Trav& T,
                                           uint32_t type, uint32_t count, uint32_t first, double tmax, LocalCounters& lc) {
    Hit& best = T.best;
    float& best_tf = T.best_tf; float& best_up = T.best_up;
    if (type == LGB_PRIM_TRIANGLE) {
        for (uint32_t i = 0; i < count; i++) {
            const uint32_t idx = first + i;
            const float4* tp = S.tri + 3 * (size_t)idx;
            const float4 q0 = __ldg(tp), q1 = __ldg(tp + 1), q2 = __ldg(tp + 2);
            if (STATS) lc.filter[2]++;
            const bool pass = f.kz == 0 ? tri_filter<0>(q0, q1, q2, f, best_tf) : f.kz == 1 ? tri_filter<1>(q0, q1, q2, f, best_tf) : tri_filter<2>(q0, q1, q2, f, best_tf);
            if (!pass) continue;
            if (STATS) lc.exact[2]++;
            double t, b0, b1, b2;
            if (triangle_exact(d3(q0.x, q0.y, q0.z), d3(q1.x, q1.y, q1.z), d3(q2.x, q2.y, q2.z), ray, t, b0, b1, b2)) {
                const uint32_t ref = LGB_PRIM_REF(LGB_PRIM_TRIANGLE, idx);
                if (ANYHIT) { if (t < tmax) { best.t = t; best.ref = ref; return true; } }
                else if (accepts<INST>(S, f, world, best, t, ref, T.tied)) { best.t = t; best.ref = ref; best_tf = __double2float_ru(t); best_up = inflate_up(t); }
            }
        }
    } else if (type == LGB_PRIM_SPHERE) {
        for (uint32_t i = 0; i < count; i++) {
            const uint32_t idx = first + i;
            const float4 s = __ldg(&S.sph32[idx]);
            if (STATS) lc.filter[0]++;
            float lx = s.x - f.ox, ly = s.y - f.oy, lz = s.z - f.oz;
            float bq = lx * f.dx + ly * f.dy + lz * f.dz;
            float tc = bq * f.inv_dd;
            float wx = __fmaf_rn(-tc, f.dx, lx), wy = __fmaf_rn(-tc, f.dy, ly), wz = __fmaf_rn(-tc, f.dz, lz);
            float perp2 = wx * wx + wy * wy + wz * wz;
            float rr = s.w + 2.0f * f.err;
            if (perp2 > rr * rr * (1.0f + 1e-6f)) continue;
            float half = rr * f.inv_len;
            float slack = fabsf(tc) * 2e-6f + 2.0f * f.err * f.inv_len;
            if (tc - half - slack > best_tf) continue;
            if (tc + half + slack < 0.0f) continue;
            if (STATS) lc.exact[0]++;
            const double2 c01 = __ldg(reinterpret_cast<const double2*>(S.sph64 + 4 * (size_t)idx));
            const double2 c23 = __ldg(reinterpret_cast<const double2*>(S.sph64 + 4 * (size_t)idx + 2));
            double t; bool inside;
            if (sphere_exact(d3(c01.x, c01.y, c23.x), c23.y, ray, t, inside)) {
                const uint32_t ref = LGB_PRIM_REF(LGB_PRIM_SPHERE, idx);
                if (ANYHIT) { if (t < tmax) { best.t = t; best.ref = ref; return true; } }
                else if (accepts<INST>(S, f, world, best, t, ref, T.tied)) { best.t = t; best.ref = ref; best_tf = __double2float_ru(t); best_up = inflate_up(t); }
            }
        }
    } else {
        for (uint32_t i = 0; i < count; i++) {
            const uint32_t idx = first + i;
            const float4 lo = __ldg(&S.cub32[2 * idx]), hi = __ldg(&S.cub32[2 * idx + 1]);
            if (STATS) lc.filter[1]++;
            float tn;
            if (!slab2(lo.x, lo.y, lo.z, hi.x, hi.y, hi.z, f, CUDART_INF_F, tn)) continue;
            if (STATS) lc.exact[1]++;
            double mn[3], mx[3];
#pragma unroll
            for (int k = 0; k < 3; k++) { mn[k] = __ldg(&S.cub64[6 * (size_t)idx + k]); mx[k] = __ldg(&S.cub64[6 * (size_t)idx + 3 + k]); }
            double t; int ua, va;
            if (cuboid_exact(mn, mx, ray, t, ua, va)) {
                const uint32_t ref = LGB_PRIM_REF(LGB_PRIM_CUBOID, idx);
                if (ANYHIT) { if (t < tmax) { best.t = t; best.ref = ref; return true; } }
                else if (accepts<INST>(S, f, world, best, t, ref, T.tied)) { best.t = t; best.ref = ref; best_tf = __double2float_ru(t); best_up = inflate_up(t); }
            }
        }
    }
    return false;
}

// The two halves of leaf_prims for ONE primitive, for the camera-grid walk (k_cprimary): a lane first runs
// filters down its list until one passes, then the warp meets for the exact f64 test.  In the fused form a warp ran the exact test
// -- by far the longest stretch of the loop body -- in nearly every iteration for whichever lanes happened to pass in that one.
// the filter of one primitive given its f32 record (sphere: q0 = {c, r}; cuboid: q0, q1 = padded lo, hi; triangle: q0..q2 = vertices)
template <bool STATS>
__device__ __forceinline__ bool prim_filter_rec(const RayF& f, float best_tf, uint32_t type, const float4 q0, const float4 q1, const float4 q2, LocalCounters& lc) {
    if (type == LGB_PRIM_SPHERE) {
        const float4 s = q0;
        if (STATS) lc.filter[0]++;
        const float lx = s.x - f.ox, ly = s.y - f.oy, lz = s.z - f.oz;
        const float bq = lx * f.dx + ly * f.dy + lz * f.dz;
        const float tc = bq * f.inv_dd;
        const float wx = __fmaf_rn(-tc, f.dx, lx), wy = __fmaf_rn(-tc, f.dy, ly), wz = __fmaf_rn(-tc, f.dz, lz);
        const float perp2 = wx * wx + wy * wy + wz * wz;
        const float rr = s.w + 2.0f * f.err;
        if (perp2 > rr * rr * (1.0f + 1e-6f)) return false;
        const float half = rr * f.inv_len;
        const float slack = fabsf(tc) * 2e-6f + 2.0f * f.err * f.inv_len;
        if (tc - half - slack > best_tf) return false;
        if (tc + half + slack < 0.0f) return false;
        return true;
    }
    if (type == LGB_PRIM_TRIANGLE) {
        if (STATS) lc.filter[2]++;
        return f.kz == 0 ? tri_filter<0>(q0, q1, q2, f, best_tf) : f.kz == 1 ? tri_filter<1>(q0, q1, q2, f, best_tf) : tri_filter<2>(q0, q1, q2, f, best_tf);
    }
    if (STATS) lc.filter[1]++;
    float tn;
    return slab2(q0.x, q0.y, q0.z, q1.x, q1.y, q1.z, f, CUDART_INF_F, tn);
}
__device__ __forceinline__ void prim_record(const DevScene& S, uint32_t type, uint32_t idx, float4& q0, float4& q1, float4& q2) {
    if (type == LGB_PRIM_SPHERE) q0 = __ldg(&S.sph32[idx]);
    else if (type == LGB_PRIM_TRIANGLE) { const float4* tp = S.tri + 3 * (size_t)idx; q0 = __ldg(tp); q1 = __ldg(tp + 1); q2 = __ldg(tp + 2); }
    else { q0 = __ldg(&S.cub32[2 * idx]); q1 = __ldg(&S.cub32[2 * idx + 1]); }
}
template <bool STATS>
__device__ __forceinline__ bool prim_filter(const DevScene& S, const RayF& f, float best_tf, uint32_t type, uint32_t idx, LocalCounters& lc) {
    float4 q0, q1 = make_float4(0.f, 0.f, 0.f, 0.f), q2 = q1;
    prim_record(S, type, idx, q0, q1, q2);
    return prim_filter_rec<STATS>(f, best_tf, type, q0, q1, q2, lc);
}
template <bool ANYHIT, bool STATS>
__device__ __forceinline__ bool prim_exact(const DevScene& S, const Ray64& world, const Ray64& ray, const RayF& f, Trav& T, uint32_t type, uint32_t idx, double tmax,
                                           LocalCounters& lc) {
    Hit& best = T.best;
    double t; bool ok;
    if (type == LGB_PRIM_SPHERE) {
        if (STATS) lc.exact[0]++;
        const double2 c01 = __ldg(reinterpret_cast<const double2*>(S.sph64 + 4 * (size_t)idx));
        const double2 c23 = __ldg(reinterpret_cast<const double2*>(S.sph64 + 4 * (size_t)idx + 2));
        bool inside;
        ok = sphere_exact(d3(c01.x, c01.y, c23.x), c23.y, ray, t, inside);
    } else if (type == LGB_PRIM_TRIANGLE) {
        if (STATS) lc.exact[2]++;
        const float4* tp = S.tri + 3 * (size_t)idx;
        const float4 q0 = __ldg(tp), q1 = __ldg(tp + 1), q2 = __ldg(tp + 2);
        double b0, b1, b2;
        ok = triangle_exact(d3(q0.x, q0.y, q0.z), d3(q1.x, q1.y, q1.z), d3(q2.x, q2.y, q2.z), ray, t, b0, b1, b2);
    } else {
        if (STATS) lc.exact[1]++;
        double mn[3], mx[3];
#pragma unroll
        for (int k = 0; k < 3; k++) { mn[k] = __ldg(&S.cub64[6 * (size_t)idx + k]); mx[k] = __ldg(&S.cub64[6 * (size_t)idx + 3 + k]); }
        int ua, va;
        ok = cuboid_exact(mn, mx, ray, t, ua, va);
    }
    if (!ok) return false;
    const uint32_t ref = LGB_PRIM_REF(type, idx);
    if (ANYHIT) { if (t < tmax) { best.t = t; best.ref = ref; return true; } return false; }
    if (accepts<false>(S, f, world, best, t, ref, T.tied)) { best.t = t; best.ref = ref; T.best_tf = __double2float_ru(t); T.best_up = inflate_up(t); }
    return false;
}

// Runs until the ray is finished (returns true; T.cur == kDone) or, with REFILL, until fewer than
// `refill_below` lanes of the warp are still traversing (returns false).  Every caller passes 0: a warp takes new
// rays only once all its lanes are done (topping it up earlier was measured slower, DESIGN.md §6).  The REFILL
// form stays because the persistent kernels schedule differently without it.
// INST (scenes with transformed aggregates): `ray` / `f` are the ray in the CURRENT space and change when the
// traversal enters or leaves a nested level; `world` is the ray as cast.  A leaf of type LGB_PRIM_INSTANCE lists child
// spaces; entering one defers the rest of the leaf and an exit marker (count field 31, payload = space to return to).
constexpr uint32_t kInstLeaf = kLeafBit | ((uint32_t)LGB_PRIM_INSTANCE << 29);
constexpr uint32_t kExitMarker = kInstLeaf | (31u << 24);
template <bool ANYHIT, bool STATS, bool REFILL, bool INST, bool SHIFT = false>
__device__ __forceinline__ bool trav_run(const DevScene& S, const Ray64& world, Ray64& ray, RayF& f, Trav& T, uint32_t* stack, float* tstack, double tmax,
                                         LocalCounters& lc, int refill_below, unsigned octw, double t0 = 0.0) {
    Hit& best = T.best;
    float& best_tf = T.best_tf; float& best_up = T.best_up;
    uint32_t& cur = T.cur; int& sp = T.sp;
    for (;;) {
        switch (INST ? f.oct : octw) {   // octw is warp-uniform: the octant shared by every ray of the warp, or 8 (mixed)
        case 0: node_loop<0, STATS, !ANYHIT>(S, f, best_up, cur, sp, stack, tstack, lc); break;
        case 1: node_loop<1, STATS, !ANYHIT>(S, f, best_up, cur, sp, stack, tstack, lc); break;
        case 2: node_loop<2, STATS, !ANYHIT>(S, f, best_up, cur, sp, stack, tstack, lc); break;
        case 3: node_loop<3, STATS, !ANYHIT>(S, f, best_up, cur, sp, stack, tstack, lc); break;
        case 4: node_loop<4, STATS, !ANYHIT>(S, f, best_up, cur, sp, stack, tstack, lc); break;
        case 5: node_loop<5, STATS, !ANYHIT>(S, f, best_up, cur, sp, stack, tstack, lc); break;
        case 6: node_loop<6, STATS, !ANYHIT>(S, f, best_up, cur, sp, stack, tstack, lc); break;
        case 7: node_loop<7, STATS, !ANYHIT>(S, f, best_up, cur, sp, stack, tstack, lc); break;
        default: node_loop<8, STATS, !ANYHIT>(S, f, best_up, cur, sp, stack, tstack, lc); break;
        }
        if (cur == kDone) return true;
        {
            const uint32_t type = (cur >> 29) & 3u, count = ((cur >> 24) & 31u) + 1u, first = cur & kLeafFirstMask;
            if (INST && type == LGB_PRIM_INSTANCE) {
                if (count == 32u) {                                   // exit marker: the nested level is done
                    T.space = first;
                    ray = ray_to_space(S, first, world);
                    f = SHIFT ? make_rayf(ray, S.spaces[first].err_abs, t0) : make_rayf(ray, S.spaces[first].err_abs);
                } else {
                    if (count > 1u) { if (!ANYHIT) tstack[sp] = -CUDART_INF_F; stack[sp] = kInstLeaf | ((count - 2u) << 24) | (first + 1u); sp++; }
                    if (!ANYHIT) tstack[sp] = -CUDART_INF_F;
                    stack[sp] = kExitMarker | T.space; sp++;
                    const uint32_t child = __ldg(&S.inst_space[first]);
                    const DevSpace& c = S.spaces[child];
                    if (!(c.flags & kSpaceIdentity)) ray = ray_into(c, ray);
                    f = SHIFT ? make_rayf(ray, c.err_abs, t0) : make_rayf(ray, c.err_abs);
                    T.space = child;
                    cur = c.root_node;
                    continue;
                }
            } else if (leaf_prims<ANYHIT, STATS, INST>(S, world, ray, f, T, type, count, first, tmax, lc)) { cur = kDone; return true; }
        }
        cur = stack_pop<!ANYHIT>(sp, stack, tstack, best_up);
        if (REFILL && __popc(__activemask()) < refill_below) return cur == kDone;
    }
}

// First ray of a traversal: the world ray in space 0 (the root aggregate may itself be transformed).
template <bool INST, bool SHIFT = false>
__device__ __forceinline__ void enter_root(const DevScene& S, const Ray64& world, Ray64& ray, RayF& f, Trav& T, double tmax, double t0 = 0.0) {
    ray = world;
    float err = S.err_abs;
    uint32_t root = 0;
    if (INST) {
        const DevSpace& s0 = S.spaces[0];
        if (!(s0.flags & kSpaceIdentity)) ray = ray_into(s0, world);
        err = s0.err_abs; root = s0.root_node;
    }
    f = SHIFT ? make_rayf(ray, err, t0) : make_rayf(ray, err);
    T.init(tmax, root);
}
template <bool ANYHIT, bool STATS, bool INST, bool SHIFT = false>
__device__ Hit traverse(const DevScene& S, const Ray64& world, double tmax, LocalCounters& lc, double t0 = 0.0) {
    Ray64 ray; RayF f; Trav T;
    enter_root<INST, SHIFT>(S, world, ray, f, T, tmax, t0);
    uint32_t stack[kStackDepth];      // depth is bounded at scene creation (lgb_api.cu), so pushes are unchecked
    float tstack[ANYHIT ? 1 : kStackDepth];
    trav_run<ANYHIT, STATS, false, INST, SHIFT>(S, world, ray, f, T, stack, tstack, tmax, lc, 0, 8u, t0);
    return T.best;
}

// ------------------------------------------------------------------ surface record of the winner
struct Surf {
    D3 g_dpdu, g_dpdv, s_dpdu, s_dpdv, n;
    bool has_n;
    uint32_t material, id;
};

// Re-derives the reference's RayIntersection for the closest primitive (sphere.rs:88-120,
// cuboid.rs:97-99, triangle.rs:257-304).  The sphere differentials use sin(theta) = sqrt(1 - cos^2)
// and cos/sin(phi) = p.xy / |p.xy| instead of acos/atan2/sin/cos (same vectors up to rounding).
__device__ void surface_of(const DevScene& S, const Ray64& ray, uint32_t ref, double& t, Surf& sf) {
    const uint32_t type = ref >> 30, idx = ref & 0x3FFFFFFFu;
    const double PI = 3.14159265358979323846264338327950288;
    sf.has_n = false; sf.n = d3(0, 0, 0);
    if (type == LGB_PRIM_SPHERE) {
        D3 c = d3(S.sph64[4 * (size_t)idx], S.sph64[4 * (size_t)idx + 1], S.sph64[4 * (size_t)idx + 2]);
        double rad = S.sph64[4 * (size_t)idx + 3];
        bool inside; double tt;
        sphere_exact(c, rad, ray, tt, inside);
        t = tt;
        D3 p = ray.o + ray.d * tt - c;
        if (p.x == 0.0 && p.y == 0.0) p.x = 1e-5 * rad;
        double rho = sqrt(p.x * p.x + p.y * p.y);
        double cphi = p.x / rho, sphi = p.y / rho;
        double cz = fmin(fmax(p.z / rad, -1.0), 1.0);
        double sth = sqrt(fmax(1.0 - cz * cz, 0.0));
        D3 dpdu = d3(-2.0 * PI * p.y, 2.0 * PI * p.x, 0.0);
        D3 dpdv = PI * d3(p.z * cphi, p.z * sphi, -rad * sth);
        if (!inside) { D3 tmp = dpdu; dpdu = dpdv; dpdv = tmp; }
        sf.g_dpdu = dpdu; sf.g_dpdv = dpdv; sf.s_dpdu = dpdu; sf.s_dpdv = dpdv;
        sf.material = S.sph_mat[idx]; sf.id = S.sph_id[idx];
    } else if (type == LGB_PRIM_CUBOID) {
        double mn[3], mx[3];
        for (int k = 0; k < 3; k++) { mn[k] = S.cub64[6 * (size_t)idx + k]; mx[k] = S.cub64[6 * (size_t)idx + 3 + k]; }
        int ua = 1, va = 2; double tt = t;
        cuboid_exact(mn, mx, ray, tt, ua, va);
        t = tt;
        D3 du = axis_vec(ua), dv = axis_vec(va);
        sf.g_dpdu = du; sf.g_dpdv = dv; sf.s_dpdu = du; sf.s_dpdv = dv;
        sf.has_n = true; sf.n = face_forward(cross(du, dv), -ray.d);
        sf.material = S.cub_mat[idx]; sf.id = S.cub_id[idx];
    } else {
        const float4 q0 = S.tri[3 * (size_t)idx], q1 = S.tri[3 * (size_t)idx + 1], q2 = S.tri[3 * (size_t)idx + 2];
        D3 p0 = d3(q0.x, q0.y, q0.z), p1 = d3(q1.x, q1.y, q1.z), p2 = d3(q2.x, q2.y, q2.z);
        const uint32_t ni = __float_as_uint(q2.w);
        double tt = t, b0 = 0, b1 = 0, b2 = 0;
        if (ni != kNoNormals) { triangle_exact(p0, p1, p2, ray, tt, b0, b1, b2); t = tt; }     // only the interpolated normal needs the barycentrics (t is the caller's, bit for bit)
        D3 dp02 = p0 - p2, dp12 = p1 - p2;
        // default uvs (0,0) (1,0) (1,1): determinant 1, dpdu = -dp02 + dp12, dpdv = dp12 (triangle.rs:258-270)
        D3 dpdu = (-1.0 * dp02 - -1.0 * dp12) * 1.0;
        D3 dpdv = (-0.0 * dp02 - -1.0 * dp12) * 1.0;
        sf.g_dpdu = dpdu; sf.g_dpdv = dpdv; sf.s_dpdu = dpdu; sf.s_dpdv = dpdv;
        sf.has_n = true;
        if (ni != kNoNormals) {                                        // triangle.rs:284-299
            const float* nn = S.tri_nrm + 9 * (size_t)ni;
            D3 n0 = d3(nn[0], nn[1], nn[2]), n1 = d3(nn[3], nn[4], nn[5]), n2 = d3(nn[6], nn[7], nn[8]);
            D3 ns = b0 * n0 + b1 * n1 + b2 * n2;
            D3 ss = dpdu;
            D3 ts = cross(ns, ss);
            if (dot(ts, ts) > 0.0) ss = cross(ts, ns); else coordinate_system(ns, ss, ts);
            sf.n = ns; sf.s_dpdu = ss; sf.s_dpdv = ts;
        } else {                                                       // triangle.rs:300-304
            sf.n = face_forward(cross(dp02, dp12), -ray.d);
        }
        sf.material = __float_as_uint(q1.w); sf.id = __float_as_uint(q0.w);
    }
}

// The local record taken back to world space, level by level from the innermost space outwards:
// transform_ray_intersection (transform.rs:243-264) then swap_backface (surface.rs:88-99, bvh.rs:510-518).
__device__ __noinline__ void record_to_world(const DevSpace* spaces, uint32_t space, Surf& sf) {
    for (uint32_t s = space; s != kNoParent; s = spaces[s].parent) {
        const DevSpace& sp = spaces[s];
        if (!(sp.flags & kSpaceIdentity)) {
            const bool shading_differs = sf.g_dpdu.x != sf.s_dpdu.x || sf.g_dpdu.y != sf.s_dpdu.y || sf.g_dpdu.z != sf.s_dpdu.z ||
                                         sf.g_dpdv.x != sf.s_dpdv.x || sf.g_dpdv.y != sf.s_dpdv.y || sf.g_dpdv.z != sf.s_dpdv.z;
            sf.g_dpdu = m4_apply(sp.m, sf.g_dpdu, 0.0); sf.g_dpdv = m4_apply(sp.m, sf.g_dpdv, 0.0);
            if (shading_differs) { sf.s_dpdu = m4_apply(sp.m, sf.s_dpdu, 0.0); sf.s_dpdv = m4_apply(sp.m, sf.s_dpdv, 0.0); }
            else { sf.s_dpdu = sf.g_dpdu; sf.s_dpdv = sf.g_dpdv; }               // RayIntersection::new, surface.rs:57-62
            if (sf.has_n) {                                                      // transform_normal, transform.rs:203-210
                const double* mi = sp.minv; const D3 n = sf.n;
                sf.n = d3(mi[0] * n.x + mi[1] * n.y + mi[2] * n.z, mi[4] * n.x + mi[5] * n.y + mi[6] * n.z, mi[8] * n.x + mi[9] * n.y + mi[10] * n.z);
            }
        }
        if (sp.flags & kSpaceSwap) {
            D3 tmp = sf.g_dpdu; sf.g_dpdu = sf.g_dpdv; sf.g_dpdv = tmp;
            tmp = sf.s_dpdu; sf.s_dpdu = sf.s_dpdv; sf.s_dpdv = tmp;
            if (sf.has_n) sf.n = -sf.n;
        }
    }
}

// ------------------------------------------------------------------ BSDF (bsdf.rs:73-92, bxdf/*)
// f64 throughout.  The reference evaluates the anisotropic Trowbridge-Reitz forms with alpha_x = alpha_y =
// roughness (plastic.rs:31-33); with equal alphas cos^2(phi) + sin^2(phi) = 1 drops out, so the device
// evaluates the isotropic closed forms (same zero / infinity guards, results equal up to f64 rounding):
//   D(wh)     = alpha^2 / (pi (alpha^2 cos^2 + sin^2)^2)                    microfacet.rs:31-40
//   Lambda(w) = (sqrt(1 + alpha^2 tan^2) - 1) / 2                           microfacet.rs:55-66
//   F         = dielectric(wi.wh, 1, 1.5) with both ratios over one divisor  fresnel.rs:37-64
//   f         = kd / pi + ks D F / (4 cos_i cos_o (1 + Lambda_o + Lambda_i)) microfacet.rs:101-115
__device__ __forceinline__ double dielectric(double cos_i) {                  // eta_i = 1, eta_t = 1.5
    cos_i = fmin(fmax(cos_i, -1.0), 1.0);
    double eta_i = 1.0, eta_t = 1.5, ratio = 1.0 / 1.5;
    if (!(cos_i > 0.0)) { eta_i = 1.5; eta_t = 1.0; ratio = 1.5; cos_i = fabs(cos_i); }
    const double sin_i = sqrt(fmax(1.0 - cos_i * cos_i, 0.0));
    const double sin_t = ratio * sin_i;
    if (sin_t >= 1.0) return 1.0;
    const double cos_t = sqrt(fmax(1.0 - sin_t * sin_t, 0.0));
    const double a = eta_t * cos_i - eta_i * cos_t, b = eta_t * cos_i + eta_i * cos_t;   // r_parl = a / b
    const double c = eta_i * cos_i - eta_t * cos_t, d = eta_i * cos_i + eta_t * cos_t;   // r_perp = c / d
    const double ad = a * d, cb = c * b, bd = b * d;
    return (ad * ad + cb * cb) / (bd * bd) * 0.5;
}
__device__ __forceinline__ double tr_lambda(double alpha2, D3 w) {
    const double c2 = w.z * w.z, s2 = fmax(1.0 - c2, 0.0);
    const double t2 = s2 / c2;
    if (isinf(t2)) return 0.0;
    return (sqrt(1.0 + alpha2 * t2) - 1.0) * 0.5;
}
// Per-hit part of the BSDF: everything that depends on wo only is evaluated once for the L + 1 evaluations
// of integrate.rs:47-67.
struct Bsdf {
    D3 ng, ns, ss, ts, kd_pi, ks, wo_l;
    double alpha2, wo_ng, cos_o, lambda_o;
    bool diffuse, glossy;
    // GENERAL variants only (dead, and removed by the compiler, in the plastic fast path): the material record as stored
    uint32_t flags; D3 c0, c1; double p0, p1, p2;
};
__device__ __forceinline__ void bsdf_prepare(Bsdf& B, D3 wo) {
    B.wo_ng = dot(wo, B.ng);
    B.wo_l = d3(dot(wo, B.ss), dot(wo, B.ts), dot(wo, B.ns));
    B.cos_o = fabs(B.wo_l.z);
    B.lambda_o = B.glossy ? tr_lambda(B.alpha2, B.wo_l) : 0.0;
}
__device__ __forceinline__ D3 bsdf_f(const Bsdf& B, D3 wi) {
    const bool reflect = dot(wi, B.ng) * B.wo_ng > 0.0;
    D3 f = d3(0, 0, 0);
    if (B.wo_l.z == 0.0) return f;
    if (!reflect) return f;                 // every lobe on this path is REFLECTION (bxdf/mod.rs:145-147)
    if (B.diffuse) f = B.kd_pi;                                                  // diffuse.rs:14
    if (B.glossy) {                                                              // microfacet.rs:101-115
        const D3 wi_l = d3(dot(wi, B.ss), dot(wi, B.ts), dot(wi, B.ns));
        const double cos_i = fabs(wi_l.z);
        const D3 wh = wi_l + B.wo_l;
        const double hh = dot(wh, wh);
        if (!(cos_i == 0.0 || B.cos_o == 0.0) && hh != 0.0) {
            const double inv = rsqrt(hh);
            const double whz = wh.z * inv;
            const double c2 = whz * whz, s2 = fmax(1.0 - c2, 0.0);
            if (c2 != 0.0) {                                                     // tan^2 infinite: D = 0
                const double F = dielectric(dot(wi_l, wh) * inv);
                const double q = B.alpha2 * c2 + s2;
                const double PI = 3.14159265358979323846264338327950288;
                const double den = PI * (q * q) * (4.0 * cos_i * B.cos_o) * (1.0 + B.lambda_o + tr_lambda(B.alpha2, wi_l));
                f = f + B.ks * (B.alpha2 * F / den);
            }
        }
    }
    return f;
}

// ---- the lobes outside the plastic fast path (SURVEY 8f item 4), in the reference's own operation order
// bxdf/mod.rs:234-258 (shading-space trigonometry)
__device__ __forceinline__ double g_sin_theta(D3 w) { return sqrt(fmax(1.0 - w.z * w.z, 0.0)); }
__device__ __forceinline__ double g_cos_phi(D3 w) { const double s = g_sin_theta(w); return s == 0.0 ? 1.0 : fmin(fmax(w.x / s, -1.0), 1.0); }
__device__ __forceinline__ double g_sin_phi(D3 w) { const double s = g_sin_theta(w); return s == 0.0 ? 0.0 : fmin(fmax(w.y / s, -1.0), 1.0); }
// fresnel.rs:37-64 for any pair of indices
__device__ __forceinline__ double dielectric_general(double cos_i, double eta_i, double eta_t) {
    cos_i = fmin(fmax(cos_i, -1.0), 1.0);
    if (!(cos_i > 0.0)) { const double tmp = eta_i; eta_i = eta_t; eta_t = tmp; cos_i = fabs(cos_i); }
    const double sin_i = sqrt(fmax(1.0 - cos_i * cos_i, 0.0));
    const double sin_t = eta_i / eta_t * sin_i;
    if (sin_t >= 1.0) return 1.0;
    const double cos_t = sqrt(fmax(1.0 - sin_t * sin_t, 0.0));
    const double r_parl = ((eta_t * cos_i) - (eta_i * cos_t)) / ((eta_t * cos_i) + (eta_i * cos_t));
    const double r_perp = ((eta_i * cos_i) - (eta_t * cos_t)) / ((eta_i * cos_i) + (eta_t * cos_t));
    return (r_parl * r_parl + r_perp * r_perp) * 0.5;
}
// fresnel.rs:68-90 with eta_i = 1 (metal.rs:21: x / 1.0 is exact)
__device__ __forceinline__ double conductor_channel(double cos_i, double eta, double k) {
    const double cos2 = cos_i * cos_i, sin2 = 1.0 - cos2;
    const double e2 = eta * eta, ek2 = k * k;
    const double t0 = e2 - ek2 - sin2;
    const double a2b2 = sqrt(t0 * t0 + 4.0 * (e2 * ek2));
    const double t1 = a2b2 + cos2;
    const double a = sqrt(0.5 * (a2b2 + t0));
    const double t2 = 2.0 * cos_i * a;
    const double rs = (t1 - t2) / (t1 + t2);
    const double t3 = cos2 * a2b2 + sin2 * sin2;
    const double t4 = t2 * sin2;
    const double rp = rs * (t3 - t4) / (t3 + t4);
    return 0.5 * (rp + rs);
}
// microfacet.rs:31-66, anisotropic
__device__ __forceinline__ double tr_d_aniso(double ax, double ay, D3 wh) {
    const double c2 = wh.z * wh.z;
    const double t2 = fmax(1.0 - c2, 0.0) / c2;
    if (isinf(t2)) return 0.0;
    const double PI = 3.14159265358979323846264338327950288;
    const double cp = g_cos_phi(wh), sp = g_sin_phi(wh);
    const double e = ((cp * cp) / (ax * ax) + (sp * sp) / (ay * ay)) * t2;
    return 1.0 / (PI * ax * ay * (c2 * c2) * (1.0 + e) * (1.0 + e));
}
__device__ __forceinline__ double tr_lambda_aniso(double ax, double ay, D3 w) {
    const double att = fabs(g_sin_theta(w) / w.z);
    if (isinf(att)) return 0.0;
    const double cp = g_cos_phi(w), sp = g_sin_phi(w);
    const double alpha = sqrt((cp * cp) * ax * ax + (sp * sp) * ay * ay);
    const double a2t2 = (alpha * att) * (alpha * att);
    return (sqrt(1.0 + a2t2) - 1.0) / 2.0;
}
// BSDF::f (bsdf.rs:73-92) for matte(sigma > 0) and metal; the lobes of glass and mirror scatter only through sample_f (mod.rs:172)
__device__ __noinline__ D3 bsdf_f_general(const Bsdf& B, D3 wi) {
    const D3 zero = d3(0, 0, 0);
    const bool reflect = dot(wi, B.ng) * B.wo_ng > 0.0;
    if (B.wo_l.z == 0.0 || !reflect) return zero;        // both lobes are REFLECTION
    const D3 wo = B.wo_l, wl = d3(dot(wi, B.ss), dot(wi, B.ts), dot(wi, B.ns));
    const uint32_t kind = B.flags >> 8;
    const double FRAC_1_PI = 0.318309886183790671537767526745028724;
    if (kind == LGB_MAT_MATTE) {                          // diffuse.rs:36-56 (Oren-Nayar, A = p1, B = p2)
        const double sin_i = g_sin_theta(wl), sin_o = g_sin_theta(wo);
        double max_cos = 0.0;
        if (sin_i > 1e-4 && sin_o > 1e-4) max_cos = fmax(g_cos_phi(wl) * g_cos_phi(wo) + g_sin_phi(wl) * g_sin_phi(wo), 0.0);
        double sin_alpha, tan_beta;
        if (fabs(wl.z) > fabs(wo.z)) { sin_alpha = sin_o; tan_beta = sin_i / fabs(wl.z); }
        else { sin_alpha = sin_i; tan_beta = sin_o / fabs(wo.z); }
        return B.c0 * FRAC_1_PI * (B.p1 + B.p2 * max_cos * sin_alpha * tan_beta);
    }
    if (kind == LGB_MAT_METAL) {                          // microfacet.rs:101-115 with Substance::Conductor (metal.rs:17-26)
        const double cos_o = fabs(wo.z), cos_i = fabs(wl.z);
        D3 wh = wl + wo;
        if (cos_i == 0.0 || cos_o == 0.0) return zero;
        if (wh.x == 0.0 && wh.y == 0.0 && wh.z == 0.0) return zero;
        wh = normalize(wh);
        const double ci = fmin(fmax(dot(wl, wh), -1.0), 1.0);
        const D3 F = d3(conductor_channel(ci, B.c0.x, B.c1.x), conductor_channel(ci, B.c0.y, B.c1.y), conductor_channel(ci, B.c0.z, B.c1.z));
        const double D = tr_d_aniso(B.p0, B.p1, wh);
        const double G = 1.0 / (1.0 + tr_lambda_aniso(B.p0, B.p1, wo) + tr_lambda_aniso(B.p0, B.p1, wl));
        return F * (D * G) / (4.0 * cos_i * cos_o);
    }
    return zero;
}
// BSDF::sample_f (bsdf.rs:94-140) for the two flag sets of integrate.rs:85,110 at sample (0.5, 0.5): a material has at most one lobe
// matching either, so comp = 0 and the pdf is the lobe's own (1 for both specular lobes).  Returns false where the sample is void.
// specular.rs:17-25 (reflection) and :44-66 (transmission); spectrum clamped to [0, 1] (bsdf.rs:122).
__device__ __forceinline__ double clamp01(double v) { return fmin(fmax(v, 0.0), 1.0); }
__device__ __forceinline__ bool sample_specular_reflection(const Bsdf& B, D3& spectrum, D3& wi_world) {
    const uint32_t kind = B.flags >> 8;
    if (kind == LGB_MAT_GLASS) { if (B.c0.x == 0.0 && B.c0.y == 0.0 && B.c0.z == 0.0) return false; }   // glass.rs:36: no reflection lobe
    else if (kind != LGB_MAT_MIRROR) return false;
    if (B.wo_l.z == 0.0) return false;
    const D3 wi = d3(-B.wo_l.x, -B.wo_l.y, B.wo_l.z);
    const double F = kind == LGB_MAT_GLASS ? dielectric_general(wi.z, 1.0, B.p0) : 1.0;
    const double ac = fabs(wi.z);
    spectrum = d3(clamp01(F * B.c0.x / ac), clamp01(F * B.c0.y / ac), clamp01(F * B.c0.z / ac));
    wi_world = d3(B.ss.x * wi.x + B.ts.x * wi.y + B.ns.x * wi.z, B.ss.y * wi.x + B.ts.y * wi.y + B.ns.y * wi.z, B.ss.z * wi.x + B.ts.z * wi.y + B.ns.z * wi.z);
    return true;
}
__device__ __forceinline__ bool sample_specular_transmission(const Bsdf& B, D3& spectrum, D3& wi_world) {
    if ((B.flags >> 8) != LGB_MAT_GLASS || (B.c1.x == 0.0 && B.c1.y == 0.0 && B.c1.z == 0.0)) return false;      // glass.rs:46
    if (B.wo_l.z == 0.0) return false;
    const bool entering = B.wo_l.z > 0.0;
    const double eta_i = entering ? 1.0 : B.p0, eta_t = entering ? B.p0 : 1.0;
    const double eta = eta_i / eta_t;
    // refract(wo, (0, 0, 1), eta), bxdf/mod.rs:164-174
    const double cos_i = 0.0 * B.wo_l.x + 0.0 * B.wo_l.y + 1.0 * B.wo_l.z;
    const double sin2_i = fmax(1.0 - cos_i * cos_i, 0.0);
    const double sin2_t = eta * eta * sin2_i;
    if (sin2_t >= 1.0) return false;
    const double cos_t = sqrt(1.0 - sin2_t);
    const double k = eta * cos_i - cos_t;
    const D3 wi = d3((eta * -1.0) * B.wo_l.x + k * 0.0, (eta * -1.0) * B.wo_l.y + k * 0.0, (eta * -1.0) * B.wo_l.z + k * 1.0);
    const double T = 1.0 - dielectric_general(wi.z, 1.0, B.p0);
    const double ac = fabs(wi.z);
    spectrum = d3(clamp01(B.c1.x * T / ac), clamp01(B.c1.y * T / ac), clamp01(B.c1.z * T / ac));
    wi_world = d3(B.ss.x * wi.x + B.ts.x * wi.y + B.ns.x * wi.z, B.ss.y * wi.x + B.ts.y * wi.y + B.ns.y * wi.z, B.ss.z * wi.x + B.ts.z * wi.y + B.ns.z * wi.z);
    return true;
}

__device__ __forceinline__ double lerp64(double t, double a, double b) { return a * (1.0 - t) + b * t; }
__device__ __forceinline__ D3 background_of(const DevShade& sh, D3 d) {                  // background.rs:25-34
    const D3 dn = normalize(d);
    const double dz = fabs(0.0 * dn.x + 0.0 * dn.y + 1.0 * dn.z);
    const double t = fmin(sqrt(1.0 - dz * dz) / sh.bg_scale, 1.0);
    return d3(lerp64(t, sh.bg_inner[0], sh.bg_outer[0]), lerp64(t, sh.bg_inner[1], sh.bg_outer[1]), lerp64(t, sh.bg_inner[2], sh.bg_outer[2]));
}

// Flags of the material of a closest hit (lgb_types.cuh) without forming its surface record.
__device__ __forceinline__ uint32_t material_flags(const DevScene& S, uint32_t ref) {
    const uint32_t type = ref >> 30, i = ref & 0x3FFFFFFFu;
    const uint32_t m = type == LGB_PRIM_SPHERE ? S.sph_mat[i] : type == LGB_PRIM_CUBOID ? S.cub_mat[i] : __float_as_uint(S.tri[3 * (size_t)i + 1].w);
    return (uint32_t)__double_as_longlong(S.materials[kMatStride * (size_t)m + 7]);
}

// Everything the lighting loop needs about the closest hit (SurfaceInteraction::from, surface.rs:158-183,
// + Material::scattering, plastic.rs:20-37 / matte.rs:18-26).
struct ShadePoint { D3 wo, ng, ns, ps, pt; Bsdf B; uint32_t mat; };

template <bool WITH_BSDF, bool INST, bool GENERAL = false>
__device__ __forceinline__ void shade_point(const DevScene& S, const Ray64& ray, double t, uint32_t ref, ShadePoint& P, uint32_t& id) {
    Surf sf; double t_again = t;
    if (INST) {                      // the record is formed in the primitive's own space, then brought back (bvh.rs:508-518)
        const uint32_t space = space_of(S, ref);
        const Ray64 local = ray_to_space(S, space, ray);
        surface_of(S, local, ref, t_again, sf);
        record_to_world(S.spaces, space, sf);
    } else surface_of(S, ray, ref, t_again, sf);
    id = sf.id;
    P.mat = sf.material;
    P.wo = -normalize(ray.d);
    P.ng = face_forward(normalize(cross(sf.g_dpdu, sf.g_dpdv)), P.wo);
    P.ns = sf.has_n ? normalize(sf.n) : normalize(cross(sf.s_dpdu, sf.s_dpdv));
    const double err = 2.220446049250313e-16 * 65536.0;        // EPSILON * 2^16, surface.rs:168
    D3 p = ray.o + ray.d * t;
    D3 p_err = P.ng * err;
    P.ps = p + p_err;                                          // integrate.rs:40
    if (GENERAL) P.pt = p - p_err;                             // origin of a transmitted ray, integrate.rs:126
    if (!WITH_BSDF) return;
    P.B.ng = P.ng; P.B.ns = P.ns; P.B.ss = normalize(sf.s_dpdu); P.B.ts = cross(P.ns, P.B.ss);
    const double* M = S.materials + kMatStride * (size_t)sf.material;
    P.B.kd_pi = d3(M[0], M[1], M[2]) * 0.318309886183790671537767526745028724; P.B.alpha2 = M[3] * M[3]; P.B.ks = d3(M[4], M[5], M[6]);
    const uint32_t flags = (uint32_t)__double_as_longlong(M[7]);
    P.B.diffuse = flags & kMatDiffuse; P.B.glossy = flags & kMatGlossy;
    if (GENERAL) { P.B.flags = flags; P.B.c0 = d3(M[0], M[1], M[2]); P.B.c1 = d3(M[4], M[5], M[6]); P.B.p0 = M[3]; P.B.p1 = M[8]; P.B.p2 = M[9]; }
    bsdf_prepare(P.B, P.wo);
}

// ------------------------------------------------------------------ lean surface record (scenes without transformed aggregates)
// For spheres, cuboids and triangles without vertex normals the reference's ng and ns (surface.rs:158-183 on the differentials of
// sphere.rs:88-120, cuboid.rs:97-99, triangle.rs:257-304) are both +-n, n the unit vector along
//   sphere    p - c            cross(dpdu, dpdv) = -+2 pi^2 rho (p - c), swapped for hits from outside (sphere.rs:117-119)
//   cuboid    e_k              the axis not among (u_axis, v_axis)
//   triangle  cross(p0 - p2, p1 - p2)
// and the signs are two of the reference's own decisions: ns = -n for a sphere hit from inside, ns = ff(n, -d) for cuboids and
// triangles (cuboid.rs:98, triangle.rs:303), ng = ff(n, wo) always (surface.rs:165).  k_setup takes those decisions (in the reference's
// arithmetic where a sign could hinge on rounding: anything within 1e-9 of a tie goes the long way through shade_point) and hands
// them to k_shade in one byte per slot, so neither kernel forms the differentials, and the unit normal costs one reciprocal
// square root instead of three normalisations.  n agrees with the reference's vectors to rounding (1e-16; 1e-11 for spheres, whose
// hit point is that far off the surface): the shadow origin p + ng 2^-36 (surface.rs:168, integrate.rs:40) needs ng to 1e-4 to come
// out bit-identical, which the occlusion-bit parity of every test confirms.
constexpr uint32_t kSfNsFlip = 1u, kSfNgFlip = 2u, kSfAxisShift = 2u, kSfGeneric = 0x80u;
struct LeanSurf { D3 n; uint32_t material, flags; };

// Unit n of the hit primitive.  EXACT_SIGNS (k_setup): also the flip bits, or kSfGeneric where the lean form does not apply.
template <bool EXACT_SIGNS>
__device__ __forceinline__ void lean_surface(const DevScene& S, const Ray64& ray, double t, uint32_t ref, uint32_t flags_in, LeanSurf& L) {
    const uint32_t type = ref >> 30, idx = ref & 0x3FFFFFFFu;
    uint32_t flags = flags_in;
    if (type == LGB_PRIM_SPHERE) {
        const double2 c01 = __ldg(reinterpret_cast<const double2*>(S.sph64 + 4 * (size_t)idx));
        const double2 c23 = __ldg(reinterpret_cast<const double2*>(S.sph64 + 4 * (size_t)idx + 2));
        const D3 c = d3(c01.x, c01.y, c23.x);
        D3 pl = ray.o + ray.d * t - c;                                  // sphere.rs:88-91
        if (pl.x == 0.0 && pl.y == 0.0) pl.x = 1e-5 * c23.y;            // sphere.rs:95
        L.material = __ldg(&S.sph_mat[idx]);
        if (EXACT_SIGNS) {
            // inside <=> the smaller root is negative (sphere.rs:57-63) <=> c = |o - c|^2 - r^2 < 0 for an accepted hit: the roots are
            // q / a and c / q (math.rs:21-27), of opposite sign iff c < 0; c == 0 is left to the reference's own sequence
            const D3 l = ray.o - c;
            const double cc = dot(l, l) - c23.y * c23.y;
            const double side = -dot(pl, ray.d);                        // ng = ff(+-n, wo): sign of n . (-d)
            const double tie = 1e-9 * (fabs(pl.x) + fabs(pl.y) + fabs(pl.z)) * (fabs(ray.d.x) + fabs(ray.d.y) + fabs(ray.d.z));
            if (cc == 0.0 || !(fabs(side) > tie) || !(c23.y > 0.0)) flags = kSfGeneric;
            else flags = (cc < 0.0 ? kSfNsFlip : 0u) | (side < 0.0 ? kSfNgFlip : 0u);
        }
        // the reference's normal is cross(dpdu, dpdv) of sphere.rs:97-116 = -+2 pi^2 (x s, y s, z rho), s = r sin(theta) = sqrt(r^2 - z^2) as the
        // clamped acos / sin pair gives it, rho = |(x, y)|: NOT the radial direction when the hit point sits 1e-10 r off the surface (a ray
        // from far away: math.rs:7-30 cancels ten digits).  Its length is rho r, so n = (x s / (rho r), y s / (rho r), z / r).
        const double A = fmax(fma(c23.y, c23.y, -(pl.z * pl.z)), 0.0), B = fma(pl.x, pl.x, pl.y * pl.y);
        const double inv_r = fast_rcp(fabs(c23.y));
        if (A > 0.0 && B > 0.0) {
            const double k = A * fast_rsqrt(A * B) * inv_r;             // s / (rho r)
            L.n = d3(pl.x * k, pl.y * k, fmin(fmax(pl.z * inv_r, -1.0), 1.0));
        } else L.n = d3(0.0, 0.0, pl.z < 0.0 ? -1.0 : 1.0);
    } else if (type == LGB_PRIM_CUBOID) {
        L.material = __ldg(&S.cub_mat[idx]);
        if (EXACT_SIGNS) {
            double mn[3], mx[3];
#pragma unroll
            for (int k = 0; k < 3; k++) { mn[k] = __ldg(&S.cub64[6 * (size_t)idx + k]); mx[k] = __ldg(&S.cub64[6 * (size_t)idx + 3 + k]); }
            // which face (cuboid.rs:63-93 keeps the axis of the winning slab): the one the hit point lies on.  The distance to the nearest
            // face plane is rounding-sized along that axis only, unless the point sits on an edge -- those go the long way.
            const D3 p = ray.o + ray.d * t;
            double e[3], scale = 0.0;
#pragma unroll
            for (int k = 0; k < 3; k++) {
                const double pk = comp(p, k);
                e[k] = fmin(fabs(pk - mn[k]), fabs(pk - mx[k]));
                scale = fmax(scale, fmax(fabs(mn[k]), fabs(mx[k])));
            }
            const int k = e[0] <= e[1] ? (e[0] <= e[2] ? 0 : 2) : (e[1] <= e[2] ? 1 : 2);
            const double second = k == 0 ? fmin(e[1], e[2]) : k == 1 ? fmin(e[0], e[2]) : fmin(e[0], e[1]);
            const double dk = comp(ray.d, k);
            // cross(e_u, e_v) = +-e_k; face-forwarded to -d (cuboid.rs:98) and to wo (surface.rs:165) it is -sign(d_k) e_k either way
            if (dk == 0.0 || !(second > 1e-6 * (1.0 + scale)) || !(e[k] < 1e-9 * (1.0 + scale))) flags = kSfGeneric;
            else flags = (dk > 0.0 ? (kSfNsFlip | kSfNgFlip) : 0u) | ((uint32_t)k << kSfAxisShift);
        }
        L.n = axis_vec((int)((flags >> kSfAxisShift) & 3u));
    } else {
        const float4* tp = S.tri + 3 * (size_t)idx;
        const float4 q0 = __ldg(tp), q1 = __ldg(tp + 1), q2 = __ldg(tp + 2);
        L.material = __float_as_uint(q1.w);
        const D3 p2 = d3(q2.x, q2.y, q2.z);
        const D3 dp02 = d3(q0.x, q0.y, q0.z) - p2, dp12 = d3(q1.x, q1.y, q1.z) - p2;
        const D3 c = fcross(dp02, dp12);
        if (EXACT_SIGNS) {
            const double side = -dot(c, ray.d);                         // n = ff(c, -d) (triangle.rs:303); ng = ff(-c^, wo): the same sign
            const double tie = 1e-9 * (fabs(c.x) + fabs(c.y) + fabs(c.z)) * (fabs(ray.d.x) + fabs(ray.d.y) + fabs(ray.d.z));
            if (__float_as_uint(q2.w) != kNoNormals || !(fabs(side) > tie)) flags = kSfGeneric;
            else flags = side < 0.0 ? (kSfNsFlip | kSfNgFlip) : 0u;
        }
        L.n = c * fast_rsqrt(fdot(c, c));
    }
    L.flags = flags;
}

// ------------------------------------------------------------------ work mapping
// n / d for the per-launch divisors (samples per pixel, supersampling root, macro tiles per row) as one 64 x 64 -> high 64 multiply:
// m = ceil(2^64 / d) (DevWork, host side) is exact for every 32-bit n (the error term n (m d - 2^64) / (d 2^64) < 2^-32 <= 1 / d);
// m == 0 stands for d == 1.  A hardware-less u32 division is ~20 instructions, and these kernels did six to eight per thread.
__device__ __forceinline__ uint32_t fdiv(uint32_t n, uint64_t m) { return m ? (uint32_t)__umul64hi((uint64_t)n, m) : n; }
// Slot indices fit 32 bits (run_capture rejects launches of 2^32 samples or more): no 64-bit divisions on this path.
__device__ __forceinline__ bool slot_to_pixel(const DevWork& W, uint64_t p64, uint32_t& x, uint32_t& y) {
    const uint32_t p = (uint32_t)p64;
    if (W.mode == 0) {
        uint32_t tile_local = p / (uint32_t)(kMacroTile * kMacroTile);
        uint32_t q = p % (uint32_t)(kMacroTile * kMacroTile);
        uint32_t tile = W.tile_list[tile_local];
        uint32_t micro = q / 32, in = q % 32;
        uint32_t px = (micro % (kMacroTile / kMicroW)) * kMicroW + in % kMicroW;
        uint32_t py = (micro / (kMacroTile / kMicroW)) * kMicroH + in / kMicroW;
        const uint32_t ty = fdiv(tile, W.fd_nmx);
        x = (tile - ty * W.n_macro_x) * kMacroTile + px;
        y = ty * kMacroTile + py;
        return x < W.w && y < W.h;
    } else {
        const uint64_t off64 = W.sub_k + (uint64_t)p * (uint64_t)W.sub_n;             // lib.rs:152-154
        if (off64 >= (uint64_t)W.w * W.h) return false;                              // (w * h < 2^32)
        const uint32_t off = (uint32_t)off64;
        y = off / W.w;
        x = off - y * W.w;
        return true;
    }
}

// camera.rs:113-146 for sample s of pixel (x, y)
__device__ __forceinline__ Ray64 camera_ray(const DevCamera& C, const DevWork& W, uint32_t x, uint32_t y, uint32_t s) {
    const D3 up = d3(C.up[0], C.up[1], C.up[2]), aux = d3(C.aux[0], C.aux[1], C.aux[2]);
    const double iph = C.image_plane_height;
    const double sox = ((double)x * W.winv - 0.5) * W.cam_ipw;
    const double soy = (0.5 - (double)(y + 1) * W.hinv) * iph;
    Ray64 r;
    r.o = d3(C.origin[0], C.origin[1], C.origin[2]) + (soy * C.pixel_separation * up) + (sox * C.pixel_separation * aux);
    const D3 d = d3(C.view[0], C.view[1], C.view[2]) + (soy * up) + (sox * aux);
    const D3 updiff = d3(W.cam_updiff[0], W.cam_updiff[1], W.cam_updiff[2]), auxdiff = d3(W.cam_auxdiff[0], W.cam_auxdiff[1], W.cam_auxdiff[2]);
    const D3 halfdiff = d3(W.cam_halfdiff[0], W.cam_halfdiff[1], W.cam_halfdiff[2]);     // (host-side, lgb_api.cu set_camera_constants)
    const uint32_t si = fdiv(s, W.fd_root);
    const double fi = (double)si, fj = (double)(s - si * C.root);
    r.d = d + (fj * updiff) + (fi * auxdiff) + halfdiff;
    return r;
}

__device__ __forceinline__ unsigned long long warp_sum(unsigned long long v) {
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xFFFFFFFFu, v, o);
    return v;
}

#ifndef LGB_MIN_BLOCKS
#define LGB_MIN_BLOCKS 10             // persistent traversal kernels at 8 / 10 / 12 blocks of 128 (64 / 48 / 40 registers): cornell 1.05 / 0.94 / 0.96 ms, simple 0.38 / 0.37 / 0.38, mixed4k through the BVH 36.1 / 36.0 / 36.0
#endif
#ifndef LGB_TRAV_THREADS
#define LGB_TRAV_THREADS 128          // threads per block of the persistent traversal kernels (256 x 4 blocks: the same on large frames, `mesh1m` 0.85 -> 0.68 ms: shorter tails)
#endif

// ================================================================== wavefront pipeline
// k_primary  persistent warps pull 32 consecutive sample slots: camera ray -> closest hit -> (t, ref)
// k_setup    per slot: miss -> background radiance; hit -> shadow origin ps and, per light, whether the
//            light can contribute at all (bsdf.rs:75: wi and wo on the same side of ng); those rays are
//            appended to that light's queue with one warp-aggregated atomic
// k_shadow   per light, persistent warps over a compacted queue: any-hit traversal to t < 1; run on queue A (the
//            centre sample of every pixel, whose occluder is remembered) and on queue C
// k_pretest  per light: the other samples try the remembered occluder first (one exact test); survivors -> queue C
// k_shade    per slot: BSDF evaluation for the unoccluded lights + ambient -> radiance (integrate.rs:47-67)
// k_resolve  per pixel: in-order sample sum, weight, quantise, uchar4 store (integrate.rs:16-20, img.rs:56-67)

template <bool RAYBUF = false>
__device__ __forceinline__ bool slot_ray(const DevCamera& C, const DevWork& W, uint64_t g, Ray64& ray, uint32_t& x, uint32_t& y, uint32_t& s) {
    if (RAYBUF) {                                                  // a level of the specular ray trees: the rays are stored
        if (g >= W.hole_lo && g < W.hole_hi) return false;
        const double* r = W.rays + 6 * g;
        ray.o = d3(r[0], r[1], r[2]); ray.d = d3(r[3], r[4], r[5]);
        x = (uint32_t)g; y = 0; s = 0;
        return true;
    }
    const uint32_t g32 = (uint32_t)g, p = fdiv(g32, W.fd_spp);
    s = g32 - p * W.spp;
    if (!slot_to_pixel(W, p, x, y)) return false;
    ray = camera_ray(C, W, x, y, s);
    return true;
}


// Warp-level work fetch for the persistent kernels: every lane whose `need` is set receives the index of a
// fresh work item (or >= total when the queue is drained) with one atomic per warp.
template <class CounterT>
__device__ __forceinline__ unsigned long long warp_fetch(CounterT* counter, bool need, unsigned lane) {
    const unsigned m = __ballot_sync(0xFFFFFFFFu, need);
    if (!m) return ~0ull;
    const int leader = __ffs(m) - 1;
    unsigned long long base = 0;
    if ((int)lane == leader) base = (unsigned long long)atomicAdd(counter, (CounterT)__popc(m));
    base = __shfl_sync(0xFFFFFFFFu, base, leader);
    return need ? base + __popc(m & ((1u << lane) - 1u)) : ~0ull;
}


// Order-preserving append of one block's items to a global queue: per-warp counts in shared memory, an
// exclusive scan over the warps, ONE global atomic per block and queue (same-address atomics serialise, and a
// warp-by-warp append would interleave the warps of different blocks, which destroys ray coherence downstream).
// Every thread of the block must call it (it synchronises); `mine` marks the threads that append `value`.
#ifndef LGB_APPEND_THREADS
#define LGB_APPEND_THREADS 512
#endif
constexpr int kAppendThreads = LGB_APPEND_THREADS;
struct AppendScratch { uint32_t warp_off[kAppendThreads / 32]; uint32_t base; };
__device__ __forceinline__ void block_append(AppendScratch& sc, bool mine, uint32_t value, uint32_t* queue, uint32_t* count) {
    const unsigned lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    const unsigned m = __ballot_sync(0xFFFFFFFFu, mine);
    if (lane == 0) sc.warp_off[warp] = __popc(m);
    __syncthreads();
    if (threadIdx.x < 32) {
        const unsigned nw = blockDim.x >> 5;
        const uint32_t c = lane < nw ? sc.warp_off[lane] : 0u;
        uint32_t incl = c;
        for (int o = 1; o < 32; o <<= 1) { const uint32_t v = __shfl_up_sync(0xFFFFFFFFu, incl, o); if ((int)lane >= o) incl += v; }
        const uint32_t tot = __shfl_sync(0xFFFFFFFFu, incl, 31);
        uint32_t base = 0;
        if (lane == 0 && tot) base = atomicAdd(count, tot);
        if (lane == 0) sc.base = base;
        if (lane < nw) sc.warp_off[lane] = incl - c;
    }
    __syncthreads();
    if (mine) queue[sc.base + sc.warp_off[warp] + __popc(m & ((1u << lane) - 1u))] = value;
    __syncthreads();          // scratch is reused by the next call
}

// The same for N consecutive items per thread (thread t holds items N t .. N t + N - 1 of the block's range): one scan and one atomic
// for N times the items, queue order = item order.
template <int N>
__device__ __forceinline__ void block_append_n(AppendScratch& sc, unsigned mine, const uint32_t* values, uint32_t* queue, uint32_t* count) {
    const unsigned lane = threadIdx.x & 31u, warp = threadIdx.x >> 5, below = (1u << lane) - 1u;
    unsigned before = 0, wtot = 0;
#pragma unroll
    for (int k = 0; k < N; k++) { const unsigned m = __ballot_sync(0xFFFFFFFFu, (mine >> k) & 1u); before += __popc(m & below); wtot += __popc(m); }
    if (lane == 0) sc.warp_off[warp] = wtot;
    __syncthreads();
    if (threadIdx.x < 32) {
        const unsigned nw = blockDim.x >> 5;
        const uint32_t c = lane < nw ? sc.warp_off[lane] : 0u;
        uint32_t incl = c;
        for (int o = 1; o < 32; o <<= 1) { const uint32_t v = __shfl_up_sync(0xFFFFFFFFu, incl, o); if ((int)lane >= o) incl += v; }
        const uint32_t tot = __shfl_sync(0xFFFFFFFFu, incl, 31);
        uint32_t base = 0;
        if (lane == 0 && tot) base = atomicAdd(count, tot);
        if (lane == 0) sc.base = base;
        if (lane < nw) sc.warp_off[lane] = incl - c;
    }
    __syncthreads();
    uint32_t at = sc.base + sc.warp_off[warp] + before;
#pragma unroll
    for (int k = 0; k < N; k++) if ((mine >> k) & 1u) queue[at++] = values[k];
    __syncthreads();          // scratch is reused by the next call
}

// The same for up to 2 x LGB_MAX_LIGHTS queues at once (k_setup: one pass over the block instead of one per queue).
// flags: bit q set <=> this thread appends `value` to queue q (queue words: V.queue / V.queue_count index q' = map[q]).
struct MultiAppendScratch { uint32_t warp_off[2 * LGB_MAX_LIGHTS][kAppendThreads / 32]; uint32_t base[2 * LGB_MAX_LIGHTS]; };
__device__ __forceinline__ void block_append_multi(MultiAppendScratch& sc, uint32_t nq, unsigned long long flags, uint32_t value,
                                                   uint32_t* queues, uint64_t queue_stride, uint32_t* counts, const uint32_t* qmap) {
    const unsigned lane = threadIdx.x & 31u, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    for (uint32_t q = 0; q < nq; q++) {
        const unsigned m = __ballot_sync(0xFFFFFFFFu, (flags >> q) & 1ull);
        if (lane == 0) sc.warp_off[q][warp] = __popc(m);
    }
    __syncthreads();
    for (uint32_t q = warp; q < nq; q += nw) {               // warp q (and q + nw, ...) scans the per-warp counts of queue q
        const uint32_t c = lane < nw ? sc.warp_off[q][lane] : 0u;
        uint32_t incl = c;
        for (int o = 1; o < 32; o <<= 1) { const uint32_t v = __shfl_up_sync(0xFFFFFFFFu, incl, o); if ((int)lane >= o) incl += v; }
        const uint32_t tot = __shfl_sync(0xFFFFFFFFu, incl, 31);
        if (lane == 0) sc.base[q] = tot ? atomicAdd(&counts[qmap[q]], tot) : 0u;
        if (lane < nw) sc.warp_off[q][lane] = incl - c;
    }
    __syncthreads();
    for (uint32_t q = 0; q < nq; q++) {
        const bool mine = (flags >> q) & 1ull;
        const unsigned m = __ballot_sync(0xFFFFFFFFu, mine);
        if (mine) queues[(size_t)qmap[q] * queue_stride + sc.base[q] + sc.warp_off[q][warp] + __popc(m & ((1u << lane) - 1u))] = value;
    }
}

template <bool STATS, bool INST, bool RAYBUF = false>
__global__ void __launch_bounds__(LGB_TRAV_THREADS, LGB_MIN_BLOCKS) k_primary(DevScene S, DevCamera C, DevWork W, DevOut O, DevWave V) {
    const uint64_t total = W.slot_list ? (W.n_list_dev ? (uint64_t)*W.n_list_dev : W.n_list) : W.n_pixels * W.spp;   // every sample slot, or the listed ones
    const unsigned lane = threadIdx.x & 31u;
    LocalCounters lc = {};
    unsigned int hits = 0, primary = 0;
    uint32_t stack[kStackDepth];
    float tstack[kStackDepth];
    Ray64 world, ray; RayF f; Trav T;      // INST: `ray` is the ray in the current space; otherwise it stays equal to `world`
    uint64_t g = 0;
    bool active = false, drained = false;
    for (;;) {
        // refill: lanes without a ray take the next sample slots
        if (!drained) {
            const unsigned idle = __ballot_sync(0xFFFFFFFFu, !active);
            if (idle == 0xFFFFFFFFu) {
                bool need = !active;
                while (__any_sync(0xFFFFFFFFu, need) && !drained) {
                    const unsigned long long idx = warp_fetch(V.work_counter, need, lane);
                    if (need) {
                        if (idx >= total) { need = false; }
                        else {
                            uint32_t x, y, s;
                            const uint64_t slot = W.slot_list ? W.slot_list[idx] : idx;
                            if (slot_ray<RAYBUF>(C, W, slot, world, x, y, s)) {
                                g = slot; enter_root<INST>(S, world, ray, f, T, CUDART_INF); active = true; need = false; primary++;
                            } else {
                                V.hit_t[slot] = CUDART_INF; V.hit_ref[slot] = kSlotUnused;     // pixel outside the film: take another
                            }
                        }
                    }
                    drained = __any_sync(0xFFFFFFFFu, idx != ~0ull && idx >= total);
                }
            }
        }
        const unsigned amask = __ballot_sync(0xFFFFFFFFu, active);
        if (!amask) break;
        const unsigned oct0 = __shfl_sync(0xFFFFFFFFu, f.oct, __ffs(amask) - 1);
        const unsigned octw = __all_sync(0xFFFFFFFFu, !active || f.oct == oct0) ? oct0 : 8u;
        if (active) {
            const bool done = trav_run<false, STATS, true, INST>(S, world, ray, f, T, stack, tstack, CUDART_INF, lc, 0, octw);
            if (done) {
                const bool hit = T.best.ref != LGB_MISS;
                V.hit_t[g] = hit ? T.best.t : CUDART_INF; V.hit_ref[g] = T.best.ref;
                hits += hit ? 1u : 0u;
                if (T.tied) { const uint32_t k = atomicAdd(V.tie_count, 1u); if (k < V.tie_cap) V.tie_list[k] = (uint32_t)g; }
                active = false;
            }
        }
    }
    if (O.counters && (!W.slot_list || W.n_list_dev)) {          // a re-trace of tied slots is not counted twice (beam fallback slots are new)
        unsigned long long v0 = warp_sum(primary), v1 = warp_sum(hits);
        if (lane == 0) { atomicAdd(&ctr(O)->primary_rays, v0); atomicAdd(&ctr(O)->primary_hits, v1); }
        if (STATS) {
            unsigned long long n = warp_sum(lc.node_tests);
            if (lane == 0) { atomicAdd(&ctr(O)->node_tests, n); atomicAdd(&ctr(O)->p_node_tests, n); }
            for (int k = 0; k < 3; k++) {
                unsigned long long a = warp_sum(lc.filter[k]), b = warp_sum(lc.exact[k]);
                if (lane == 0) { atomicAdd(&ctr(O)->filter[k], a); atomicAdd(&ctr(O)->exact[k], b); atomicAdd(&ctr(O)->p_filter[k], a); atomicAdd(&ctr(O)->p_exact[k], b); }
            }
        }
    }
}

// ================================================================== pixel beams
// At >= 4 samples per pixel the rays of a pixel are a thin bundle with a common origin, and each of them repeats
// almost the same interior-node tests.  k_beam traverses the BVH ONCE per pixel with the whole bundle -- a slab test
// on the per-axis interval of 1/d over the bundle, conservative for every ray in it -- and writes the leaves it
// reaches, sorted by entry distance; k_leafp then gives every sample ray only those leaves (f32 filter + exact f64
// test as everywhere else; a leaf whose entry distance is beyond the ray's best hit ends the walk).  Pixels whose
// bundle reaches more than kBeamList leaves fall back to the per-ray traversal (k_primary over a slot list).
// The bundle is described by its centre ray plus, per axis, the relative spread of 1/d over the bundle: for every ray r
// of the bundle and every plane, t_a(r) = (plane - o) / d_a(r) lies within t_a(centre) (1 -+ spread_a), because the
// origin is common.  So the bundle test is the centre ray's slab test with every entry distance taken as early and every
// exit distance as late as the spread allows: six more FMAs, and conservative for every ray of the bundle.
struct BeamF { float sx, sy, sz; };
__device__ __forceinline__ BeamF make_beam(const DevCamera& C, const DevWork& W, uint32_t x, uint32_t y, const Ray64& centre) {
    const uint32_t r = C.root;
    const uint32_t corner[4] = {0u, r - 1u, (r - 1u) * r, r * r - 1u};         // sample (i, j) = i * root + j; d is affine in (i, j)
    double dmin[3] = {CUDART_INF, CUDART_INF, CUDART_INF}, dmax[3] = {-CUDART_INF, -CUDART_INF, -CUDART_INF};
    for (int c = 0; c < 4; c++) {
        const Ray64 q = camera_ray(C, W, x, y, corner[c]);
        dmin[0] = fmin(dmin[0], q.d.x); dmax[0] = fmax(dmax[0], q.d.x);
        dmin[1] = fmin(dmin[1], q.d.y); dmax[1] = fmax(dmax[1], q.d.y);
        dmin[2] = fmin(dmin[2], q.d.z); dmax[2] = fmax(dmax[2], q.d.z);
    }
    const double dc[3] = {centre.d.x, centre.d.y, centre.d.z};
    float sp[3];
    for (int a = 0; a < 3; a++) {
        // 1/d over [dmin, dmax] relative to 1/dc; a component that changes sign inside the bundle does not constrain at all
        if (!(dmin[a] > 0.0) && !(dmax[a] < 0.0)) { sp[a] = 1e30f; continue; }
        const double lo = fmin(fabs(dmin[a]), fabs(dmax[a])), hi = fmax(fabs(dmin[a]), fabs(dmax[a])), c = fabs(dc[a]);
        const double up = c / lo - 1.0, dn = 1.0 - c / hi;                      // |1/d| in |1/dc| [1 - dn, 1 + up]
        sp[a] = __double2float_ru(fmax(fmax(up, dn), 0.0) * 1.0000001 + 4e-7);   // + the f32 rounding of the centre ray's own 1/d and products
    }
    BeamF B; B.sx = sp[0]; B.sy = sp[1]; B.sz = sp[2];
    return B;
}
// OCT: direction octant of the centre ray (bit a set <=> d[a] < 0), or 8 for the generic form.
template <int OCT>
__device__ __forceinline__ bool beam_slab(float lx, float ly, float lz, float hx, float hy, float hz, const RayF& f, const BeamF& B, float& tn_out) {
    float tnx, tfx, tny, tfy, tnz, tfz;
    if (OCT < 8) {
        tnx = __fmaf_rn((OCT & 1) ? hx : lx, f.ix, f.nx); tfx = __fmaf_rn((OCT & 1) ? lx : hx, f.ix, f.nx);
        tny = __fmaf_rn((OCT & 2) ? hy : ly, f.iy, f.ny); tfy = __fmaf_rn((OCT & 2) ? ly : hy, f.iy, f.ny);
        tnz = __fmaf_rn((OCT & 4) ? hz : lz, f.iz, f.nz); tfz = __fmaf_rn((OCT & 4) ? lz : hz, f.iz, f.nz);
    } else {
        const float ax = __fmaf_rn(lx, f.ix, f.nx), bx = __fmaf_rn(hx, f.ix, f.nx), ay = __fmaf_rn(ly, f.iy, f.ny), by = __fmaf_rn(hy, f.iy, f.ny);
        const float az = __fmaf_rn(lz, f.iz, f.nz), bz = __fmaf_rn(hz, f.iz, f.nz);
        tnx = fminf(ax, bx); tfx = fmaxf(ax, bx); tny = fminf(ay, by); tfy = fmaxf(ay, by); tnz = fminf(az, bz); tfz = fmaxf(az, bz);
    }
    // widen: entry distances down, exit distances up, by |t| * spread
    tnx = __fmaf_rn(-fabsf(tnx), B.sx, tnx); tfx = __fmaf_rn(fabsf(tfx), B.sx, tfx);
    tny = __fmaf_rn(-fabsf(tny), B.sy, tny); tfy = __fmaf_rn(fabsf(tfy), B.sy, tfy);
    tnz = __fmaf_rn(-fabsf(tnz), B.sz, tnz); tfz = __fmaf_rn(fabsf(tfz), B.sz, tfz);
    const float tn = fmaxf(fmaxf(fmaxf(tnx, tny), tnz), 0.0f);
    const float tf = fminf(fminf(tfx, tfy), tfz) * (1.0f + 9.5367431640625e-7f);
    tn_out = tn;
    return !(tn > tf);            // a NaN (inf - inf on a degenerate axis) must not reject
}

// k_beam also traces the pixel's CENTRE sample exactly while it walks (nearer child first): its closest hit t_c bounds
// the walk -- a node or leaf whose bundle entry distance exceeds B = t_c (1 + 1/32) is not visited.  The list is then
// complete for every ray of the pixel whose own closest hit is not farther than B; k_leafp sends the others (depth
// discontinuities inside the pixel) and the pixels with more than kBeamList leaves to the per-ray traversal.
#ifndef LGB_BEAM_MARGIN
#define LGB_BEAM_MARGIN 1.03125f
#endif
constexpr float kBeamMargin = LGB_BEAM_MARGIN;
#ifndef LGB_BEAM_THREADS
#define LGB_BEAM_THREADS 64          // as for k_leafp: 256 -> 64 threads per block, 54.02 -> 53.59 ms/frame
#endif
template <bool STATS>
__global__ void __launch_bounds__(LGB_BEAM_THREADS, 1024 / LGB_BEAM_THREADS) k_beam(DevScene S, DevCamera C, DevWork W, DevOut O, DevWave V) {
    const uint64_t p = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const unsigned lane = threadIdx.x & 31u;
    LocalCounters lc = {};
    unsigned int hits = 0, primary = 0;
    if (p < W.n_pixels) {
        uint32_t x, y;
        uint32_t n = 0;
        float bound = CUDART_INF_F;
        if (slot_to_pixel(W, p, x, y)) {
            const uint64_t g = p * W.spp + W.anchor;
            const Ray64 world = camera_ray(C, W, x, y, W.anchor);
            const BeamF B = make_beam(C, W, x, y, world);
            Ray64 ray; RayF f; Trav T;
            enter_root<false>(S, world, ray, f, T, CUDART_INF);
            primary++;
            uint32_t stack[kStackDepth]; float tstack[kStackDepth]; int sp = 0;
            uint2 list[kBeamList];                     // (leaf word, entry distance) in visiting order: nearer child first, so nearly sorted
            uint32_t cur = 0;
            bool over = false;
            while (cur != kDone && !over) {
                if (cur & kLeafBit) {                  // a leaf the bundle enters before the bound: list it, test the centre ray
                    // ... primitive by primitive: the bundle against the primitive's own (padded) box, so that the sample rays of
                    // the pixel are handed only the primitives their bundle can reach -- a quarter of a leaf on average
                    const uint32_t type = (cur >> 29) & 3u, count = ((cur >> 24) & 31u) + 1u, first = cur & kLeafFirstMask;
                    for (uint32_t i = 0; i < count; i++) {
                        const uint32_t idx = first + i;
                        float lx, ly, lz, hx, hy, hz;
                        if (type == LGB_PRIM_TRIANGLE) {
                            const float4* tp = S.tri + 3 * (size_t)idx;
                            const float4 q0 = __ldg(tp), q1 = __ldg(tp + 1), q2 = __ldg(tp + 2);
                            lx = fminf(q0.x, fminf(q1.x, q2.x)); hx = fmaxf(q0.x, fmaxf(q1.x, q2.x));
                            ly = fminf(q0.y, fminf(q1.y, q2.y)); hy = fmaxf(q0.y, fmaxf(q1.y, q2.y));
                            lz = fminf(q0.z, fminf(q1.z, q2.z)); hz = fmaxf(q0.z, fmaxf(q1.z, q2.z));
                        } else if (type == LGB_PRIM_SPHERE) {
                            const float4 sp4 = __ldg(&S.sph32[idx]);
                            const float rr = __fadd_ru(sp4.w, f.err);
                            lx = __fsub_rd(sp4.x, rr); hx = __fadd_ru(sp4.x, rr); ly = __fsub_rd(sp4.y, rr); hy = __fadd_ru(sp4.y, rr); lz = __fsub_rd(sp4.z, rr); hz = __fadd_ru(sp4.z, rr);
                        } else {
                            const float4 lo = __ldg(&S.cub32[2 * idx]), hi = __ldg(&S.cub32[2 * idx + 1]);      // padded already
                            lx = lo.x; ly = lo.y; lz = lo.z; hx = hi.x; hy = hi.y; hz = hi.z;
                        }
                        if (type != LGB_PRIM_CUBOID) {                                 // the padding of the node boxes (k_make_items)
                            lx = __fsub_rd(lx, f.err); ly = __fsub_rd(ly, f.err); lz = __fsub_rd(lz, f.err);
                            hx = __fadd_ru(hx, f.err); hy = __fadd_ru(hy, f.err); hz = __fadd_ru(hz, f.err);
                        }
                        float tn;
                        if (!beam_slab<8>(lx, ly, lz, hx, hy, hz, f, B, tn) || tn > bound) continue;
                        if (n == (uint32_t)kBeamList) { over = true; break; }
                        list[n++] = make_uint2(kLeafBit | (type << 29) | idx, __float_as_uint(tn));
                        leaf_prims<false, STATS, false>(S, world, ray, f, T, type, 1u, idx, CUDART_INF, lc);
                        bound = T.best_up * kBeamMargin;
                    }
                    if (over) break;
                    cur = kDone;
                } else {
                    const float4* np = S.nodes + 4 * (size_t)cur;
                    const float4 n0 = __ldg(np), n1 = __ldg(np + 1), n2 = __ldg(np + 2);
                    const float2 n3 = __ldg(reinterpret_cast<const float2*>(np + 3));
                    if (STATS) lc.node_tests++;
                    float t0, t1;
                    bool h0, h1;
                    switch (f.oct) {
#define LGB_BEAM_CASE(o) case o: h0 = beam_slab<o>(n0.x, n0.y, n0.z, n0.w, n1.x, n1.y, f, B, t0); h1 = beam_slab<o>(n1.z, n1.w, n2.x, n2.y, n2.z, n2.w, f, B, t1); break;
                    LGB_BEAM_CASE(0) LGB_BEAM_CASE(1) LGB_BEAM_CASE(2) LGB_BEAM_CASE(3) LGB_BEAM_CASE(4) LGB_BEAM_CASE(5) LGB_BEAM_CASE(6)
                    default: h0 = beam_slab<7>(n0.x, n0.y, n0.z, n0.w, n1.x, n1.y, f, B, t0); h1 = beam_slab<7>(n1.z, n1.w, n2.x, n2.y, n2.z, n2.w, f, B, t1); break;
#undef LGB_BEAM_CASE
                    }
                    h0 = h0 && t0 <= bound; h1 = h1 && t1 <= bound;
                    const uint32_t c0 = __float_as_uint(n3.x), c1 = __float_as_uint(n3.y);
                    if (h0 && h1) {
                        const bool swap = t1 < t0;
                        cur = swap ? c1 : c0;
                        tstack[sp] = swap ? t0 : t1; stack[sp++] = swap ? c0 : c1;
                    } else if (h0) cur = c0;
                    else if (h1) cur = c1;
                    else cur = kDone;
                }
                while (cur == kDone && sp) {           // nearest deferred entry that still starts before the bound
                    --sp;
                    if (tstack[sp] <= bound) cur = stack[sp];
                }
            }
            if (over) {
                n = kBeamOverflow; primary--;              // the walk was cut short: every sample of the pixel, the centre one included, is traced on its own
            } else {
                const bool hit = T.best.ref != LGB_MISS;
                V.hit_t[g] = hit ? T.best.t : CUDART_INF; V.hit_ref[g] = T.best.ref;      // the centre sample is done
                hits += hit ? 1u : 0u;
                if (T.tied) { const uint32_t k = atomicAdd(V.tie_count, 1u); if (k < V.tie_cap) V.tie_list[k] = (uint32_t)g; }
                uint32_t m = 0;
                for (uint32_t i = 0; i < n; i++) {         // entries listed before the bound tightened may lie beyond it now
                    if (__uint_as_float(list[i].y) > bound) continue;
                    V.beam_list[(size_t)m * W.n_pixels + p] = list[i]; m++;
                }
                n = m;
            }
        }
        V.beam_count[p] = n;
        V.beam_bound[p] = bound;
    }
    if (O.counters) {
        unsigned long long v0 = warp_sum(primary), v1 = warp_sum(hits);
        if (lane == 0) { atomicAdd(&ctr(O)->primary_rays, v0); atomicAdd(&ctr(O)->primary_hits, v1); }
        if (STATS) {
            const unsigned long long v = warp_sum(lc.node_tests);
            if (lane == 0) { atomicAdd(&ctr(O)->node_tests, v); atomicAdd(&ctr(O)->p_node_tests, v); atomicAdd(&ctr(O)->beam_node_tests, v); }
            for (int k = 0; k < 3; k++) {
                unsigned long long a = warp_sum(lc.filter[k]), b2 = warp_sum(lc.exact[k]);
                if (lane == 0) { atomicAdd(&ctr(O)->filter[k], a); atomicAdd(&ctr(O)->exact[k], b2); atomicAdd(&ctr(O)->p_filter[k], a); atomicAdd(&ctr(O)->p_exact[k], b2); }
            }
        }
    }
}

// One thread per sample slot (the centre sample is already done): the leaves of its pixel's beam, nearest first.
#ifndef LGB_LEAFP_THREADS
#define LGB_LEAFP_THREADS 64         // a block waits for its slowest ray before it frees its slots: 256 -> 64 threads, 55.15 -> 53.97 ms/frame
#endif
template <bool STATS>
__global__ void __launch_bounds__(LGB_LEAFP_THREADS, 1024 / LGB_LEAFP_THREADS) k_leafp(DevScene S, DevCamera C, DevWork W, DevOut O, DevWave V) {
    __shared__ AppendScratch sc;
    const uint64_t total = W.n_pixels * W.spp;
    const uint64_t g = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const unsigned lane = threadIdx.x & 31u;
    LocalCounters lc = {};
    unsigned int hits = 0, primary = 0;
    bool fallback = false;
    const uint32_t pix = fdiv((uint32_t)g, W.fd_spp);
    if (g < total && (uint32_t)g - pix * W.spp != W.anchor) {
        const uint64_t p = pix;
        const uint32_t n = V.beam_count[p];
        Ray64 world; uint32_t x, y, s;
        if (!slot_ray(C, W, g, world, x, y, s)) { V.hit_t[g] = CUDART_INF; V.hit_ref[g] = kSlotUnused; }
        else if (n == kBeamOverflow) fallback = true;
        else {
            const float bound = V.beam_bound[p];
            Ray64 ray; RayF f; Trav T;
            enter_root<false>(S, world, ray, f, T, CUDART_INF);
            for (uint32_t i = 0; i < n; i++) {
                const uint2 e = __ldg(&V.beam_list[(size_t)i * W.n_pixels + p]);
                if (__uint_as_float(e.y) > T.best_up) continue;            // starts beyond the best hit (the list is only nearly sorted)
                leaf_prims<false, STATS, false>(S, world, ray, f, T, (e.x >> 29) & 3u, ((e.x >> 24) & 31u) + 1u, e.x & kLeafFirstMask, CUDART_INF, lc);
            }
            if (T.best_up <= bound) {              // the list held every leaf that starts before the bound: the result is final
                const bool hit = T.best.ref != LGB_MISS;
                primary++;
                V.hit_t[g] = hit ? T.best.t : CUDART_INF; V.hit_ref[g] = T.best.ref;
                hits += hit ? 1u : 0u;
                if (T.tied) { const uint32_t k = atomicAdd(V.tie_count, 1u); if (k < V.tie_cap) V.tie_list[k] = (uint32_t)g; }
            } else fallback = true;                // hit beyond the bound, or none: this ray needs its own traversal
        }
    } else if (g < total) {                        // centre sample: done by k_beam, unless ...
        uint32_t x, y;
        if (!slot_to_pixel(W, pix, x, y)) { V.hit_t[g] = CUDART_INF; V.hit_ref[g] = kSlotUnused; }      // ... the pixel is outside the film
        else if (V.beam_count[pix] == kBeamOverflow) fallback = true;                                      // ... or its walk was cut short
    }
    block_append(sc, fallback, (uint32_t)g, V.fallback_list, V.fallback_count);
    if (O.counters) {
        unsigned long long v0 = warp_sum(primary), v1 = warp_sum(hits);
        if (lane == 0) { atomicAdd(&ctr(O)->primary_rays, v0); atomicAdd(&ctr(O)->primary_hits, v1); }
        if (STATS) {
            for (int k = 0; k < 3; k++) {
                unsigned long long a = warp_sum(lc.filter[k]), b = warp_sum(lc.exact[k]);
                if (lane == 0) { atomicAdd(&ctr(O)->filter[k], a); atomicAdd(&ctr(O)->exact[k], b); atomicAdd(&ctr(O)->p_filter[k], a); atomicAdd(&ctr(O)->p_exact[k], b); }
            }
        }
    }
}

// Which lights can contribute at a hit: bsdf.f is zero unless wi and wo are on the same side of ng (bsdf.rs:75,85-86) -- the light
// then adds exactly zero whether or not it is occluded, so no shadow ray is traced (DESIGN.md 4.4).  The test is the reference's own
// product with the normalised wi; its sign is that of the unnormalised dot product whenever that is clear of rounding (1e-6 of
// |v|_1), which spares the sqrt and the division.  wo_ng: dot(wo, ng), or any positive number where ng faces wo by construction.
__device__ __forceinline__ uint32_t light_gates(const DevScene& S, const Ray64& ray, D3 ps, D3 ng, double wo_ng, bool lean) {
    uint32_t gate = 0;
    for (uint32_t l = 0; l < S.n_lights; l++) {
        const double* L = S.lights + 9 * (size_t)l;
        const D3 v = d3(L[0], L[1], L[2]) - ps;
        const double dv = dot(v, ng);
        bool same;
        if (fabs(dv) > 1e-6 * (fabs(v.x) + fabs(v.y) + fabs(v.z)) && fabs(wo_ng) > 1e-100) same = (dv > 0.0) == (wo_ng > 0.0);
        else same = dot(normalize(v), ng) * (lean ? dot(-normalize(ray.d), ng) : wo_ng) > 0.0;
        if (same) gate |= 1u << l;
    }
    return gate;
}

// The rare slot whose sign decisions lean_surface leaves to the reference's own sequence (k_cprimary<SETUP>), out of line.
// Written so that nothing of the kernel's own state has its address taken: the scene record is read from global memory
// (DevScene::self), the ray goes by value, the results go straight to the slot's wavefront entries.  With
// `const DevScene& S` bound to the kernel's parameter block every thread copied the 350-byte record to its stack at entry (28 STL.64
// per thread: 30 GB of local stores per mixed4k frame, through L1 into L2), and the ray after it -- for a call one slot in a million makes.
__device__ __noinline__ void setup_generic_slot(const DevScene* Sg, double ox, double oy, double oz, double dx, double dy, double dz, double t, uint32_t ref,
                                                double* ps_out, uint32_t* gate_out) {
    const DevScene& S = *Sg;
    Ray64 ray; ray.o = d3(ox, oy, oz); ray.d = d3(dx, dy, dz);
    ShadePoint P; uint32_t id;
    shade_point<false, false>(S, ray, t, ref, P, id);
    ps_out[0] = P.ps.x; ps_out[1] = P.ps.y; ps_out[2] = P.ps.z;
    *gate_out = light_gates(S, ray, P.ps, P.ng, dot(P.wo, P.ng), false);
}
// ================================================================== primary rays through the camera grid (lgb_grid.cu)
// One thread per sample slot: the pixel's tile lists every primitive one of its samples can see, nearest first; each gets the f32
// filter + the reference's exact test (closest hit, reference-order ties as everywhere), and the walk stops at the first entry that
// starts beyond the best hit.  No traversal, no per-ray stack, no fallback: the list is complete for every ray of the tile.
#ifndef LGB_CPRIMARY_THREADS
#define LGB_CPRIMARY_THREADS 128
#endif
#ifndef LGB_CPRIMARY_BLOCKS
#define LGB_CPRIMARY_BLOCKS (1280 / LGB_CPRIMARY_THREADS)     // 8 / 10 / 12 / 14 blocks of 128 (64 / 48 / 40 / 32 registers), no staging: 5.70 / 5.54 / 5.67 / 6.10 ms on mixed4k
#endif
// SETUP (plain captures with light grids): once the walk is over the thread still holds the camera ray and the hit, and the hit
// primitive is warm in L1 -- it does k_setup's work for its slot right there (surface record, sign byte, shadow origin, gates) and
// k_setup drops out of the frame.  The walk's own state is dead by then, so nothing is added to what lives across it.
template <bool STATS, bool SETUP = false>
__global__ void __launch_bounds__(LGB_CPRIMARY_THREADS, LGB_CPRIMARY_BLOCKS) k_cprimary(DevScene S, DevCamera C, DevWork W, DevOut O, DevWave V) {
    const uint64_t total = W.n_pixels * W.spp;
    const uint64_t g = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const unsigned lane = threadIdx.x & 31u;
    LocalCounters lc = {};
    unsigned int hits = 0, primary = 0;
    bool valid = false;
    uint32_t x = 0, y = 0, s = 0;
    if (g < total) {
        const uint32_t p = fdiv((uint32_t)g, W.fd_spp);
        s = (uint32_t)g - p * W.spp;
        if (!slot_to_pixel(W, p, x, y)) { wst(&V.hit_t[g], (double)(CUDART_INF)); wst(&V.hit_ref[g], (uint32_t)(kSlotUnused)); }
        else valid = true;
    }
    const size_t cell = (size_t)(y >> W.cg_shift) * W.cg_nx + (size_t)(x >> W.cg_shift);
    uint32_t b = 0, e = 0;
    if (valid) { b = __ldg(W.cg_start + cell); e = __ldg(W.cg_start + cell + 1); }
    if (valid) {
        {
            const Ray64 world = camera_ray(C, W, x, y, s);
            Ray64 ray; RayF f; Trav T;
            enter_root<false>(S, world, ray, f, T, CUDART_INF);
            primary++;
            const float to_t = f.inv_len * (1.0f - 2e-6f);                   // an entry's distance from the eye -> a lower bound of its ray parameter
            const bool sorted = e - b <= kGridSortMax;                       // (longer lists are not sorted: lgb_grid.cu)
            // positions [b, e) are the tile's list, [e, e2) the large list (both nearest first)
            const uint32_t e2 = e + W.cg_n_large;
            for (uint32_t i = b;;) {
                uint32_t cand = 0xFFFFFFFFu;
                while (i < e2) {
                    const bool in_cell = i < e;
                    const uint2 r = __ldg(in_cell ? W.cg_entries + i : W.cg_large + (i - e));
                    i++;
                    if (__uint_as_float(r.y) * to_t > T.best_up) { if (!in_cell) i = e2; else if (sorted) i = e; continue; }    // nearest first: nothing behind the best hit can beat it
                    if (prim_filter<STATS>(S, f, T.best_tf, r.x >> 30, r.x & 0x3FFFFFFFu, lc)) { cand = r.x; break; }
                }
                if (cand == 0xFFFFFFFFu) break;
                prim_exact<false, STATS>(S, world, ray, f, T, cand >> 30, cand & 0x3FFFFFFFu, CUDART_INF, lc);
            }
            const bool hit = T.best.ref != LGB_MISS;
            wst(&V.hit_t[g], (double)(hit ? T.best.t : CUDART_INF)); wst(&V.hit_ref[g], (uint32_t)(T.best.ref));
            hits += hit ? 1u : 0u;
            if (T.tied) { const uint32_t k = atomicAdd(V.tie_count, 1u); if (k < V.tie_cap) V.tie_list[k] = (uint32_t)g; }
            if (SETUP && hit) {
                const uint32_t ref = T.best.ref; const double t = T.best.t;
                if (S.specular && (material_flags(S, ref) & kMatSpecular)) { wst(&V.occl[g], (uint32_t)(0)); wst(&V.gate[g], (uint32_t)(0)); }     // glass, mirror: BSDF::f is zero (bxdf/mod.rs:172)
                else {
                    LeanSurf Ls;
                    lean_surface<true>(S, world, t, ref, 0u, Ls);
                    if (Ls.flags & kSfGeneric) setup_generic_slot(S.self, world.o.x, world.o.y, world.o.z, world.d.x, world.d.y, world.d.z, t, ref, V.ps + 3 * g, V.gate + g);
                    else {
                        const D3 ng = (Ls.flags & kSfNgFlip) ? -Ls.n : Ls.n;
                        const D3 ps = world.o + world.d * t + ng * (2.220446049250313e-16 * 65536.0);       // surface.rs:168, integrate.rs:40
                        wst(&V.ps[3 * g + 0], ps.x); wst(&V.ps[3 * g + 1], ps.y); wst(&V.ps[3 * g + 2], ps.z);
                        wst(&V.gate[g], (uint32_t)(light_gates(S, world, ps, ng, 1.0, true)));
                    }
                    wst(&V.sflags[g], (unsigned char)((unsigned char)Ls.flags));
                    wst(&V.occl[g], (uint32_t)(0));
                }
            }
        }
    }
    if (O.counters) {
        const unsigned long long v0 = __popc(__ballot_sync(0xFFFFFFFFu, primary != 0)), v1 = __popc(__ballot_sync(0xFFFFFFFFu, hits != 0));      // (one slot per thread)
        if (lane == 0) { atomicAdd(&ctr(O)->primary_rays, v0); atomicAdd(&ctr(O)->primary_hits, v1); }
        if (STATS) {
            for (int k = 0; k < 3; k++) {
                unsigned long long a = warp_sum(lc.filter[k]), b = warp_sum(lc.exact[k]);
                if (lane == 0) { atomicAdd(&ctr(O)->filter[k], a); atomicAdd(&ctr(O)->exact[k], b); atomicAdd(&ctr(O)->p_filter[k], a); atomicAdd(&ctr(O)->p_exact[k], b); }
            }
        }
    }
}

template <bool ALL_SHADOWS, bool INST, bool RAYBUF = false>
__global__ void __launch_bounds__(kAppendThreads) k_setup(DevScene S, DevCamera C, DevShade sh, DevWork W, DevOut O, DevWave V) {
    constexpr bool LEAN = !INST && !RAYBUF;          // camera rays of scenes without transformed aggregates: lean_surface
    const uint64_t total = W.n_pixels * W.spp;
    const uint64_t g = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t need = 0;
    bool live = false;
    if (g < total) {
        const uint32_t ref = V.hit_ref[g];
        const double t_hit = V.hit_t[g];             // (requested together with ref: one round trip to memory instead of two)
        Ray64 ray; uint32_t x, y, s;
        bool ref_done = false;
        if (ref != kSlotUnused && slot_ray<RAYBUF>(C, W, g, ray, x, y, s)) {
            const uint64_t gi = ((uint64_t)y * W.w + x) * W.spp + s;
            if (ref == LGB_MISS) {                                   // the background is evaluated by k_shade
                if (O.aov_id) O.aov_id[gi] = LGB_MISS;
                if (O.aov_t) O.aov_t[gi] = CUDART_INF;
                if (O.aov_occl) O.aov_occl[gi] = 0;
            } else {
                // glass and mirror: BSDF::f is zero whatever the light does (bxdf/mod.rs:172) -- no shadow ray, no shadow origin
                if (!ALL_SHADOWS && S.specular && (material_flags(S, ref) & kMatSpecular)) { V.occl[g] = 0; V.gate[g] = 0; ref_done = true; }
            }
            if (ref != LGB_MISS && !ref_done) {
                live = true;
                const double t = t_hit;
                D3 ng, ps; double wo_ng; uint32_t sflags = kSfGeneric;
                if (LEAN) {                          // ng = +-n and the reference's sign decisions, no differentials (lean_surface)
                    LeanSurf Ls;
                    lean_surface<true>(S, ray, t, ref, 0u, Ls);
                    sflags = Ls.flags;
                    if (!(sflags & kSfGeneric)) {
                        ng = (sflags & kSfNgFlip) ? -Ls.n : Ls.n;
                        ps = ray.o + ray.d * t + ng * (2.220446049250313e-16 * 65536.0);       // surface.rs:168, integrate.rs:40
                        wo_ng = 1.0;                 // ng faces wo by construction (clear of rounding, else kSfGeneric)
                    }
                }
                if (sflags & kSfGeneric) {
                    ShadePoint P; uint32_t id;
                    shade_point<false, INST>(S, ray, t, ref, P, id);
                    ng = P.ng; ps = P.ps; wo_ng = dot(P.wo, P.ng);
                }
                V.ps[3 * g + 0] = ps.x; V.ps[3 * g + 1] = ps.y; V.ps[3 * g + 2] = ps.z;
                if (O.aov_id) O.aov_id[gi] = canonical_id(S, ref);
                if (O.aov_t) O.aov_t[gi] = t;
                const uint32_t gate = light_gates(S, ray, ps, ng, wo_ng, !(sflags & kSfGeneric));
                need = ALL_SHADOWS ? (S.n_lights >= 32u ? 0xFFFFFFFFu : (1u << S.n_lights) - 1u) : gate;
                V.occl[g] = 0;
                V.gate[g] = gate;
                if (LEAN) V.sflags[g] = (unsigned char)sflags;
            }
        }
    }
    if (S.grids) return;         // light grids (k_gshadow) read ps / gate by slot: no queues
    // compacted per-light shadow queues (A: anchor sample of the pixel, B: the others), block-ordered, all at once:
    // flag bit 2l = queue A of light l, bit 2l + 1 = queue B
    __shared__ MultiAppendScratch sc;
    __shared__ uint32_t qmap[2 * LGB_MAX_LIGHTS];
    if (threadIdx.x < 2 * S.n_lights) qmap[threadIdx.x] = (threadIdx.x >> 1) * 3 + ((threadIdx.x & 1) ? kQueueB : kQueueA);
    __syncthreads();
    const bool anchor = W.spp == 1 || (uint32_t)g - fdiv((uint32_t)g, W.fd_spp) * W.spp == W.anchor;
    unsigned long long flags = 0;
    if (live) for (uint32_t l = 0; l < S.n_lights; l++) if ((need >> l) & 1u) flags |= 1ull << (2 * l + (anchor ? 0 : 1));
    block_append_multi(sc, 2 * S.n_lights, flags, (uint32_t)g, V.queue, V.queue_stride, V.queue_count, qmap);
}

// Exact test of ONE primitive against a shadow ray: true iff the reference's intersect accepts it with t < 1
// (the same calls the traversal makes for a candidate, light/point.rs:48-49).
template <bool INST>
__device__ __forceinline__ bool occludes(const DevScene& S, uint32_t ref, const Ray64& world) {
    const uint32_t type = ref >> 30, idx = ref & 0x3FFFFFFFu;
    Ray64 ray = world;
    if (INST) ray = ray_to_space(S, space_of(S, ref), world);
    double t;
    if (type == LGB_PRIM_TRIANGLE) {
        const float4* tp = S.tri + 3 * (size_t)idx;
        const float4 q0 = __ldg(tp), q1 = __ldg(tp + 1), q2 = __ldg(tp + 2);
        double b0, b1, b2;
        return triangle_exact(d3(q0.x, q0.y, q0.z), d3(q1.x, q1.y, q1.z), d3(q2.x, q2.y, q2.z), ray, t, b0, b1, b2) && t < 1.0;
    }
    if (type == LGB_PRIM_SPHERE) {
        const double2 c01 = __ldg(reinterpret_cast<const double2*>(S.sph64 + 4 * (size_t)idx));
        const double2 c23 = __ldg(reinterpret_cast<const double2*>(S.sph64 + 4 * (size_t)idx + 2));
        bool inside;
        return sphere_exact(d3(c01.x, c01.y, c23.x), c23.y, ray, t, inside) && t < 1.0;
    }
    double mn[3], mx[3];
#pragma unroll
    for (int k = 0; k < 3; k++) { mn[k] = __ldg(&S.cub64[6 * (size_t)idx + k]); mx[k] = __ldg(&S.cub64[6 * (size_t)idx + 3 + k]); }
    int ua, va;
    return cuboid_exact(mn, mx, ray, t, ua, va) && t < 1.0;
}

// Queue B -> occl bit (blocked by the occluder the pixel's anchor ray found) or queue C (needs a traversal).
#ifndef LGB_PRETEST_ITEMS
#define LGB_PRETEST_ITEMS 2          // 1 / 2 / 4 / 8 entries per thread and round: 53.60 / 52.54 / 53.20 / 53.12 ms/frame
#endif
constexpr int kPretestItems = LGB_PRETEST_ITEMS;
template <bool INST>
__global__ void __launch_bounds__(kAppendThreads) k_pretest(DevScene S, DevWork W, DevOut O, DevWave V, uint32_t light) {
    __shared__ AppendScratch sc;
    const unsigned total = V.queue_count[light * 3 + kQueueB];
    const unsigned lane = threadIdx.x & 31u;
    const double* L = S.lights + 9 * (size_t)light;
    const D3 lp = d3(L[0], L[1], L[2]);
    unsigned ncached = 0;
    // kPretestItems consecutive queue entries per thread and round: their loads are in flight together and one block-ordered
    // append (three barriers) serves them all
    for (uint64_t i0 = (uint64_t)blockIdx.x * blockDim.x * kPretestItems; i0 < total; i0 += (uint64_t)gridDim.x * blockDim.x * kPretestItems) {      // block-uniform trip count
        const uint64_t first = i0 + threadIdx.x * kPretestItems;
        uint32_t g[kPretestItems], oc[kPretestItems];
        unsigned to_c = 0;
#pragma unroll
        for (int k = 0; k < kPretestItems; k++) {
            g[k] = 0; oc[k] = LGB_MISS;
            if (first + k < total) {
                g[k] = V.queue[(size_t)(light * 3 + kQueueB) * V.queue_stride + first + k];
                if (g[k] != kEntryDone) {                                          // (k_swalk has resolved it from the pixel's shadow beam)
                    oc[k] = V.occluder[(size_t)light * W.n_pixels + fdiv(g[k], W.fd_spp)];
                    to_c |= 1u << k;
                }
            }
        }
#pragma unroll
        for (int k = 0; k < kPretestItems; k++) {
            if (oc[k] != LGB_MISS) {
                Ray64 ray;
                ray.o = d3(V.ps[3 * (size_t)g[k]], V.ps[3 * (size_t)g[k] + 1], V.ps[3 * (size_t)g[k] + 2]);
                ray.d = lp - ray.o;                                                  // light/point.rs:43-44
                if (occludes<INST>(S, oc[k], ray)) { atomicOr(&V.occl[g[k]], 1u << light); to_c &= ~(1u << k); ncached++; }   // (another light's chain may be running on a side stream)
            }
        }
        block_append_n<kPretestItems>(sc, to_c, g, V.queue + (size_t)(light * 3 + kQueueC) * V.queue_stride, &V.queue_count[light * 3 + kQueueC]);
    }
    if (O.counters) {
        const unsigned long long n = warp_sum(ncached);
        if (lane == 0 && n) { atomicAdd(&ctr(O)->shadow_cached, n); atomicAdd(&ctr(O)->shadow_occluded, n); }
        if (blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(&ctr(O)->shadow_traced, (unsigned long long)total);
    }
}

#ifndef LGB_SBEAM_THREADS
#define LGB_SBEAM_THREADS_ 64
#else
#define LGB_SBEAM_THREADS_ LGB_SBEAM_THREADS
#endif
// ================================================================== shadow beams
// The shadow rays of a pixel towards one light are a bundle too: seen from the light they share their origin, and their
// directions (light -> shadow origin of every sample) differ by the footprint of one pixel on the surface.  k_sbeam, one thread per
// ANCHOR ray (queue A: the centre sample of a pixel) that k_shadow found FREE, walks the BVH once with that bundle over the segment
// light .. surface (parameter s in [0, 1], the reference's t = 1 - s) and lists the primitives whose own boxes the bundle meets
// (f32 only: pure culling).  Where the list is complete the other samples of the pixel need no traversal at all: k_swalk tests
// them against the listed primitives only (f32 filter + exact f64 test) and removes them from queue B.  Whatever is left (pixels
// whose anchor is blocked -- k_pretest tries its occluder on the other samples first, as before --, overflowing lists, pixels
// without an anchor ray) goes the old way: k_pretest, then k_shadow over queue C.
template <bool STATS>
__global__ void __launch_bounds__(LGB_SBEAM_THREADS_, 1024 / LGB_SBEAM_THREADS_) k_sbeam(DevScene S, DevWork W, DevOut O, DevWave V, uint32_t light,
                                                                                     uint2* list_out, uint32_t* count_out) {
    const unsigned total = V.free_count[light];                           // the anchor rays k_shadow found free (listed in queue C's space)
    const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
    const unsigned lane = threadIdx.x & 31u;
    LocalCounters lc = {};
    if (i < total) {
        const uint32_t ga = V.queue[(size_t)(light * 3 + kQueueC) * V.queue_stride + i];
        const uint32_t p = fdiv(ga, W.fd_spp);
        {
        const double* Lp = S.lights + 9 * (size_t)light;
        const D3 lp = d3(Lp[0], Lp[1], Lp[2]);
        Ray64 centre; centre.o = lp;                                      // the bundle runs from the common point towards the surface
        centre.d = d3(V.ps[3 * (size_t)ga], V.ps[3 * (size_t)ga + 1], V.ps[3 * (size_t)ga + 2]) - lp;
        // per-axis interval of the directions over the samples of the pixel that have a shadow origin
        double dmin[3] = {centre.d.x, centre.d.y, centre.d.z}, dmax[3] = {centre.d.x, centre.d.y, centre.d.z};
        for (uint32_t k = 0; k < W.spp; k++) {
            const size_t g = (size_t)p * W.spp + k;
            const uint32_t ref = V.hit_ref[g];
            if (ref == LGB_MISS || ref == kSlotUnused) continue;
            const double dx = V.ps[3 * g] - lp.x, dy = V.ps[3 * g + 1] - lp.y, dz = V.ps[3 * g + 2] - lp.z;
            dmin[0] = fmin(dmin[0], dx); dmax[0] = fmax(dmax[0], dx); dmin[1] = fmin(dmin[1], dy); dmax[1] = fmax(dmax[1], dy);
            dmin[2] = fmin(dmin[2], dz); dmax[2] = fmax(dmax[2], dz);
        }
        const double dc[3] = {centre.d.x, centre.d.y, centre.d.z};
        float sp[3];
        for (int a = 0; a < 3; a++) {                                     // as make_beam: |1/d| over the bundle relative to the centre's
            if (!(dmin[a] > 0.0) && !(dmax[a] < 0.0)) { sp[a] = 1e30f; continue; }
            const double lo = fmin(fabs(dmin[a]), fabs(dmax[a])), hi = fmax(fabs(dmin[a]), fabs(dmax[a])), c = fabs(dc[a]);
            const double up = c / lo - 1.0, dn = 1.0 - c / hi;
            sp[a] = __double2float_ru(fmax(fmax(up, dn), 0.0) * 1.0000001 + 4e-7);
        }
        BeamF B; B.sx = sp[0]; B.sy = sp[1]; B.sz = sp[2];
        const RayF f = make_rayf(centre, S.err_abs);
        const float smax = 1.0f + 1e-5f;                                  // occluders lie at s in (0, 1]; the slack covers the f32 slab arithmetic
        uint32_t stack[kStackDepth]; int sp_ = 0;
        uint2 list[kBeamList];
        uint32_t n = 0, cur = 0;
        bool over = false;
        while (cur != kDone && !over) {
            if (cur & kLeafBit) {
                const uint32_t type = (cur >> 29) & 3u, count = ((cur >> 24) & 31u) + 1u, first = cur & kLeafFirstMask;
                for (uint32_t k = 0; k < count; k++) {
                    const uint32_t idx = first + k;
                    float lx, ly, lz, hx, hy, hz;
                    if (type == LGB_PRIM_TRIANGLE) {
                        const float4* tp = S.tri + 3 * (size_t)idx;
                        const float4 q0 = __ldg(tp), q1 = __ldg(tp + 1), q2 = __ldg(tp + 2);
                        lx = fminf(q0.x, fminf(q1.x, q2.x)); hx = fmaxf(q0.x, fmaxf(q1.x, q2.x));
                        ly = fminf(q0.y, fminf(q1.y, q2.y)); hy = fmaxf(q0.y, fmaxf(q1.y, q2.y));
                        lz = fminf(q0.z, fminf(q1.z, q2.z)); hz = fmaxf(q0.z, fmaxf(q1.z, q2.z));
                    } else if (type == LGB_PRIM_SPHERE) {
                        const float4 s4 = __ldg(&S.sph32[idx]);
                        const float rr = __fadd_ru(s4.w, f.err);
                        lx = __fsub_rd(s4.x, rr); hx = __fadd_ru(s4.x, rr); ly = __fsub_rd(s4.y, rr); hy = __fadd_ru(s4.y, rr); lz = __fsub_rd(s4.z, rr); hz = __fadd_ru(s4.z, rr);
                    } else {
                        const float4 lo = __ldg(&S.cub32[2 * idx]), hi = __ldg(&S.cub32[2 * idx + 1]);
                        lx = lo.x; ly = lo.y; lz = lo.z; hx = hi.x; hy = hi.y; hz = hi.z;
                    }
                    if (type != LGB_PRIM_CUBOID) {
                        lx = __fsub_rd(lx, f.err); ly = __fsub_rd(ly, f.err); lz = __fsub_rd(lz, f.err);
                        hx = __fadd_ru(hx, f.err); hy = __fadd_ru(hy, f.err); hz = __fadd_ru(hz, f.err);
                    }
                    float tn;
                    if (!beam_slab<8>(lx, ly, lz, hx, hy, hz, f, B, tn) || tn > smax) continue;
                    if (n == (uint32_t)kBeamList) { over = true; break; }
                    list[n++] = make_uint2(kLeafBit | (type << 29) | idx, __float_as_uint(tn));
                }
                cur = kDone;
            } else {
                const float4* np = S.nodes + 4 * (size_t)cur;
                const float4 n0 = __ldg(np), n1 = __ldg(np + 1), n2 = __ldg(np + 2);
                const float2 n3 = __ldg(reinterpret_cast<const float2*>(np + 3));
                if (STATS) lc.node_tests++;
                float t0, t1;
                bool h0, h1;
                switch (f.oct) {
#define LGB_BEAM_CASE(o) case o: h0 = beam_slab<o>(n0.x, n0.y, n0.z, n0.w, n1.x, n1.y, f, B, t0); h1 = beam_slab<o>(n1.z, n1.w, n2.x, n2.y, n2.z, n2.w, f, B, t1); break;
                LGB_BEAM_CASE(0) LGB_BEAM_CASE(1) LGB_BEAM_CASE(2) LGB_BEAM_CASE(3) LGB_BEAM_CASE(4) LGB_BEAM_CASE(5) LGB_BEAM_CASE(6)
                default: h0 = beam_slab<7>(n0.x, n0.y, n0.z, n0.w, n1.x, n1.y, f, B, t0); h1 = beam_slab<7>(n1.z, n1.w, n2.x, n2.y, n2.z, n2.w, f, B, t1); break;
#undef LGB_BEAM_CASE
                }
                h0 = h0 && t0 <= smax; h1 = h1 && t1 <= smax;
                const uint32_t c0 = __float_as_uint(n3.x), c1 = __float_as_uint(n3.y);
                if (h0 && h1) { cur = c0; stack[sp_++] = c1; }
                else if (h0) cur = c0;
                else if (h1) cur = c1;
                else cur = kDone;
            }
            if (cur == kDone && sp_ && !over) cur = stack[--sp_];
        }
        if (!over) {
            for (uint32_t k = 0; k < n; k++) list_out[(size_t)k * W.n_pixels + p] = list[k];
            count_out[p] = n;                                             // complete: k_swalk serves the other samples from it
        }
        }
    }
    if (O.counters && STATS) {
        unsigned long long nt = warp_sum(lc.node_tests);
        if (lane == 0) atomicAdd(&ctr(O)->node_tests, nt);
    }
}
// One thread per queue-B entry (the non-anchor samples): where the pixel's bundle left a complete list, the ray is tested against
// the listed primitives alone, any hit with t < 1 (light/point.rs:48-49), and the entry is taken out of the queue.
#ifndef LGB_SWALK_THREADS
#define LGB_SWALK_THREADS 128        // 32 / 64 / 128 / 256 threads: 46.5 / 45.5 / 45.1 / 45.4 ms/frame
#endif
#ifndef LGB_SBEAM_THREADS
#define LGB_SBEAM_THREADS 64
#endif
template <bool STATS>
__global__ void __launch_bounds__(LGB_SWALK_THREADS, 1024 / LGB_SWALK_THREADS) k_swalk(DevScene S, DevWork W, DevOut O, DevWave V, uint32_t light,
                                                                                       const uint2* list_in, const uint32_t* count_in) {
    const unsigned total = V.queue_count[light * 3 + kQueueB];
    const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
    const unsigned lane = threadIdx.x & 31u;
    LocalCounters lc = {};
    unsigned occluded = 0;
    if (i < total) {
        uint32_t* slot = V.queue + (size_t)(light * 3 + kQueueB) * V.queue_stride + i;
        const uint32_t g = *slot;
        const uint32_t p = fdiv(g, W.fd_spp);
        const uint32_t n = count_in[p];
        if (n != kBeamOverflow) {
            const double* Lp = S.lights + 9 * (size_t)light;
            Ray64 world;
            world.o = d3(V.ps[3 * (size_t)g], V.ps[3 * (size_t)g + 1], V.ps[3 * (size_t)g + 2]);
            world.d = d3(Lp[0], Lp[1], Lp[2]) - world.o;
            Ray64 ray; RayF f; Trav T;
            enter_root<false>(S, world, ray, f, T, 1.0);
            bool hit = false;
            for (uint32_t k = 0; k < n && !hit; k++) {
                const uint2 e = __ldg(&list_in[(size_t)k * W.n_pixels + p]);
                hit = leaf_prims<true, STATS, false>(S, world, ray, f, T, (e.x >> 29) & 3u, 1u, e.x & kLeafFirstMask, 1.0, lc);
            }
            if (hit) { atomicOr(&V.occl[g], 1u << light); occluded++; }
            *slot = kEntryDone;
        }
    }
    if (O.counters) {
        unsigned long long v = warp_sum(occluded);
        if (lane == 0 && v) atomicAdd(&ctr(O)->shadow_occluded, v);
        if (STATS) {
            for (int k = 0; k < 3; k++) {
                unsigned long long a = warp_sum(lc.filter[k]), b = warp_sum(lc.exact[k]);
                if (lane == 0) { atomicAdd(&ctr(O)->filter[k], a); atomicAdd(&ctr(O)->exact[k], b); }
            }
        }
    }
}

// ================================================================== shadow rays through the light grids (lgb_grid.cu)
// One thread per sample slot, every light in turn: the ray's direction seen from the light selects ONE cell of that light's cube
// map; its entries (nearest to the light first) and the light's few large primitives get the f32 filter + the reference's exact
// test, any hit with t < 1 (light/point.rs:48-49), up to the first entry that starts beyond the ray's own length.
#ifndef LGB_GSHADOW_THREADS
#define LGB_GSHADOW_THREADS 64            // 256 / 128 / 64 threads per block at 1024 per SM: 7.35 / 6.79 / 6.69 ms on mixed4k (a block keeps its registers until its slowest ray is done)
#endif
// Registers per thread against threads per SM (mixed4k, 64-thread blocks): 80 / 72 / 64 / 48 / 40 / 32 registers = 768 / 896 / 1024 / 1280 /
// 1536 / 2048 threads: 7.53 / 6.93 / 6.69 / 6.06 / 6.01 / 7.21 ms.  The walk waits on loads; more rays in flight buy more than the spills cost.
#ifndef LGB_GSHADOW_MIN_BLOCKS
#define LGB_GSHADOW_MIN_BLOCKS (1536 / LGB_GSHADOW_THREADS)
#endif
// The shadow ray from `o` towards light l (light/point.rs:43-44: d = light - o, blocked iff the closest t < 1) against that light's grid.
template <bool STATS>
__device__ __forceinline__ bool grid_blocked(const DevScene& S, D3 o, uint32_t l, LocalCounters& lc) {
    Ray64 world;
    world.o = o;
    const double* Lp = S.lights + 9 * (size_t)l;
    world.d = d3(Lp[0], Lp[1], Lp[2]) - world.o;
    // the cell of the direction light -> surface: major axis a, u = d_b / |d_a|, v = d_c / |d_a| (as face_rect, lgb_grid.cu)
    const double ax = fabs(world.d.x), ay = fabs(world.d.y), az = fabs(world.d.z);
    const int a = ax >= ay ? (ax >= az ? 0 : 2) : (ay >= az ? 1 : 2);
    const double da = -(a == 0 ? world.d.x : a == 1 ? world.d.y : world.d.z);
    const double db = -(a == 0 ? world.d.y : a == 1 ? world.d.z : world.d.x), dc = -(a == 0 ? world.d.z : a == 1 ? world.d.x : world.d.y);
    if (da == 0.0) return false;                                       // the light sits on the shadow origin: nothing lies between
    const DevGrid* G = S.grids + l;
    const uint32_t res = __ldg(&G->res), n_large = __ldg(&G->n_large);
    const int face = 2 * a + (da < 0.0 ? 1 : 0);
    const double* map = G->map[face];                                   // the face's cells cover [u0, u0 + res / su] x [v0, v0 + res / sv]; outside clamps to the border
    const double inv = fast_rcp(fabs(da));
    const int cu = min(max((int)floor((db * inv - __ldg(map)) * __ldg(map + 1)), 0), (int)res - 1);
    const int cv = min(max((int)floor((dc * inv - __ldg(map + 2)) * __ldg(map + 3)), 0), (int)res - 1);
    const size_t cell = ((size_t)face * res + (size_t)cv) * res + (size_t)cu;
    const uint32_t* cs = G->cell_start;
    const uint32_t b = __ldg(cs + cell), e = __ldg(cs + cell + 1);
    Ray64 ray; RayF f; Trav T;
    enter_root<false>(S, world, ray, f, T, 1.0);
    const float dd = f.dx * f.dx + f.dy * f.dy + f.dz * f.dz;
    const float len_up = dd * f.inv_len * (1.0f + 1e-5f) + f.err;     // an entry that starts farther from the light than the ray does cannot block it
    bool hit = false;
    const bool sorted = e - b <= kGridSortMax;                         // (longer lists are not sorted: lgb_grid.cu)
    const uint2* en = G->entries;
    const uint2* lg = G->large;
    // The fused walk (filter and exact test in one loop body), not k_cprimary's split form: at 40-48 registers the split walk took
    // 6.02 ms against 5.75 on mixed4k.  An any-hit walk ends at its first exact hit, so there is less for the warp to converge on.
    for (uint32_t i = b; i < e && !hit; i++) {
        const uint2 r = __ldg(en + i);
        if (__uint_as_float(r.y) > len_up) { if (sorted) break; else continue; }
        hit = leaf_prims<true, STATS, false>(S, world, ray, f, T, r.x >> 30, 1u, r.x & 0x3FFFFFFFu, 1.0, lc);
    }
    for (uint32_t i = 0; i < n_large && !hit; i++) {
        const uint2 r = __ldg(lg + i);
        if (__uint_as_float(r.y) > len_up) break;
        hit = leaf_prims<true, STATS, false>(S, world, ray, f, T, r.x >> 30, 1u, r.x & 0x3FFFFFFFu, 1.0, lc);
    }
    return hit;
}

template <bool STATS, bool ALL_SHADOWS>
__global__ void __launch_bounds__(LGB_GSHADOW_THREADS, LGB_GSHADOW_MIN_BLOCKS) k_gshadow(DevScene S, DevCamera C, DevWork W, DevOut O, DevWave V) {
    const uint64_t total = W.n_pixels * W.spp;
    const uint64_t g = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const unsigned lane = threadIdx.x & 31u;
    LocalCounters lc = {};
    unsigned traced = 0, occluded = 0;
    if (g < total) {
        const uint32_t ref = wld(&V.hit_ref[g]);
        uint32_t mask = 0;
        D3 ps = d3(0, 0, 0);
        // gate and shadow origin are requested together with the hit word, not one after the other (three dependent round trips
        // were 18 % of this kernel's stall samples); for a miss they hold stale values nobody looks at
        const uint32_t gate = ALL_SHADOWS ? (S.n_lights >= 32u ? 0xFFFFFFFFu : (1u << S.n_lights) - 1u) : wld(&V.gate[g]);
        ps = d3(wld(&V.ps[3 * g]), wld(&V.ps[3 * g + 1]), wld(&V.ps[3 * g + 2]));
        if (ref != LGB_MISS && ref != kSlotUnused) mask = gate;
        if (mask) {
            uint32_t occl = 0;
            for (uint32_t l = 0; l < S.n_lights; l++) {
                if (!((mask >> l) & 1u)) continue;
                traced++;
                if (grid_blocked<STATS>(S, ps, l, lc)) { occl |= 1u << l; occluded++; }
            }
            wst(&V.occl[g], occl);
        }
    }
    if (O.counters) {
        const unsigned long long v0 = warp_sum(traced), v1 = warp_sum(occluded);
        if (lane == 0 && v0) {
            if (W.mode == 3) atomicAdd(&ctr(O)->secondary_rays, v0);      // a level of the specular ray trees: lgb_stats.secondary_rays
            else { atomicAdd(&ctr(O)->shadow_traced, v0); atomicAdd(&ctr(O)->shadow_occluded, v1); }
        }
        if (STATS) {
            for (int k = 0; k < 3; k++) {
                unsigned long long a = warp_sum(lc.filter[k]), b = warp_sum(lc.exact[k]);
                if (lane == 0) { atomicAdd(&ctr(O)->filter[k], a); atomicAdd(&ctr(O)->exact[k], b); }
            }
        }
    }
}

template <bool STATS, bool INST>
__global__ void __launch_bounds__(LGB_TRAV_THREADS, LGB_MIN_BLOCKS) k_shadow(DevScene S, DevWork W, DevOut O, DevWave V, uint32_t light, int which) {
    const unsigned total = V.queue_count[light * 3 + which];
    const uint32_t* q = V.queue + (size_t)(light * 3 + which) * V.queue_stride;
    const bool record = which == kQueueA && W.spp > 1;      // anchor rays remember their occluder for k_pretest
    const double* L = S.lights + 9 * (size_t)light;
    const D3 lp = d3(L[0], L[1], L[2]);
    const unsigned lane = threadIdx.x & 31u;
    LocalCounters lc = {};
    unsigned int occluded = 0;
    uint32_t stack[kStackDepth];
    Ray64 world, ray; RayF f; Trav T;
    uint32_t g = 0;
    bool active = false, drained = false;
    for (;;) {
        if (!drained) {
            const unsigned idle = __ballot_sync(0xFFFFFFFFu, !active);
            if (idle == 0xFFFFFFFFu) {
                const unsigned long long idx = warp_fetch(V.queue_fetch + light * 3 + which, !active, lane);
                if (!active && idx < total) {
                    g = q[idx];
                    world.o = d3(V.ps[3 * (size_t)g], V.ps[3 * (size_t)g + 1], V.ps[3 * (size_t)g + 2]);
                    world.d = lp - world.o;                                      // light/point.rs:43-44
                    enter_root<INST>(S, world, ray, f, T, 1.0); active = true;
                }
                drained = __any_sync(0xFFFFFFFFu, idx != ~0ull && idx >= total);
            }
        }
        const unsigned amask = __ballot_sync(0xFFFFFFFFu, active);
        if (!amask) break;
        const unsigned oct0 = __shfl_sync(0xFFFFFFFFu, f.oct, __ffs(amask) - 1);
        const unsigned octw = __all_sync(0xFFFFFFFFu, !active || f.oct == oct0) ? oct0 : 8u;
        if (active) {
            const bool done = trav_run<true, STATS, true, INST>(S, world, ray, f, T, stack, nullptr, 1.0, lc, 0, octw);
            if (done) {
                if (T.best.ref != LGB_MISS) { atomicOr(&V.occl[g], 1u << light); occluded++; }
                if (record) V.occluder[(size_t)light * W.n_pixels + fdiv(g, W.fd_spp)] = T.best.ref;
                if (record && W.beams && T.best.ref == LGB_MISS) {       // a free anchor: its pixel gets a shadow beam (k_sbeam); listed in queue C's space
                    const unsigned peers = __activemask(), leader = __ffs(peers) - 1;
                    uint32_t base = 0;
                    if (lane == leader) base = atomicAdd(V.free_count + light, (uint32_t)__popc(peers));
                    base = __shfl_sync(peers, base, leader);
                    V.queue[(size_t)(light * 3 + kQueueC) * V.queue_stride + base + __popc(peers & ((1u << lane) - 1u))] = g;
                }
                active = false;
            }
        }
    }
    if (O.counters) {
        unsigned long long v = warp_sum(occluded);
        if (lane == 0) atomicAdd(&ctr(O)->shadow_occluded, v);
        if (which == kQueueA && blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(&ctr(O)->shadow_traced, (unsigned long long)total);
        if (STATS) {
            unsigned long long n = warp_sum(lc.node_tests);
            if (lane == 0) atomicAdd(&ctr(O)->node_tests, n);
            for (int k = 0; k < 3; k++) {
                unsigned long long a = warp_sum(lc.filter[k]), b = warp_sum(lc.exact[k]);
                if (lane == 0) { atomicAdd(&ctr(O)->filter[k], a); atomicAdd(&ctr(O)->exact[k], b); }
            }
        }
    }
}

#ifndef LGB_SHADE_MIN_BLOCKS
#define LGB_SHADE_MIN_BLOCKS 4
#endif
#ifndef LGB_FUSED_THREADS
#define LGB_FUSED_THREADS 128u          // blocks of 256 / 128 threads (whole pixels): k_shade_lean 4.05 / 3.88 ms on mixed4k
#endif
#ifndef LGB_GSHADE_MIN_BLOCKS
#define LGB_GSHADE_MIN_BLOCKS 2      // the GENERAL variants (every material, spawn of the specular rays)
#endif
__device__ __forceinline__ uchar4 quantise(D3 c) {                     // img.rs:56-67
    uchar4 px;
    px.x = (unsigned char)round(fmin(fmax(c.x, 0.0), 1.0) * 255.0);
    px.y = (unsigned char)round(fmin(fmax(c.y, 0.0), 1.0) * 255.0);
    px.z = (unsigned char)round(fmin(fmax(c.z, 0.0), 1.0) * 255.0);
    px.w = 255;
    return px;
}
// The linear film (lgb_capture_linear): the colour quantise() would receive, rounded to nearest f32, 3 floats per pixel.
__device__ __forceinline__ void store_linear(uint8_t* film, uint64_t i, D3 c) {
    float* f = reinterpret_cast<float*>(film) + 3 * i;
    f[0] = __double2float_rn(c.x); f[1] = __double2float_rn(c.y); f[2] = __double2float_rn(c.z);
}
// Radiance of every sample slot (integrate.rs:23-80) and, FUSED (spp <= 256: a block holds whole pixels), the film:
// the samples of a pixel meet in shared memory and are summed in sample order (integrate.rs:16-20), so the
// 24 B/sample radiance buffer and k_resolve drop out.  Thread t of a block: pixel t / spp of the block, sample t % spp.
// LINEAR (FUSED only): the film is the linear f32 one (store_linear) instead of RGBA8.
// The rays below one specular hit (specular_reflect / specular_transmit, integrate.rs:82-132) appended to the next level of the
// wavefront: reflected rays fill the level's slots from 0, transmitted ones from V.next_t_base, so each kind stays with its own
// (neighbouring rays of a warp then point the same way); one record per hit tells k_gather where the children are.
__device__ __forceinline__ void spawn_children(const ShadePoint& P, const DevWave& V, uint32_t g) {
    SpawnRec rec; rec.slot = g; rec.child_r = rec.child_t = kNoChild; rec.pad = 0;
    rec.spec_r[0] = rec.spec_r[1] = rec.spec_r[2] = rec.spec_t[0] = rec.spec_t[1] = rec.spec_t[2] = rec.c = 0.0;
    Ray64 rr, rt; D3 spec, wi;
    bool has_r = false, has_t = false;
    if (sample_specular_reflection(P.B, spec, wi) && !(spec.x == 0.0 && spec.y == 0.0 && spec.z == 0.0) && !(dot(wi, P.ns) <= 0.0)) {
        has_r = true; rr.o = P.ps; rr.d = -1.0 * P.wo + 2.0 * dot(P.wo, P.ns) * P.ns;      // bxdf::util::reflect, mod.rs:160-162
        rec.spec_r[0] = spec.x; rec.spec_r[1] = spec.y; rec.spec_r[2] = spec.z;
    }
    if (sample_specular_transmission(P.B, spec, wi)) {
        const double c = fabs(dot(wi, P.ns));
        if (!(spec.x == 0.0 && spec.y == 0.0 && spec.z == 0.0) && c != 0.0) {
            has_t = true; rt.o = P.pt; rt.d = wi; rec.c = c;
            rec.spec_t[0] = spec.x; rec.spec_t[1] = spec.y; rec.spec_t[2] = spec.z;
        }
    }
    const unsigned peers = __activemask(), lane = threadIdx.x & 31u, leader = __ffs(peers) - 1;
    const unsigned mr = __ballot_sync(peers, has_r), mt = __ballot_sync(peers, has_t);
    uint32_t b_rec = 0, b_r = 0, b_t = 0;
    if (lane == leader) {
        b_rec = atomicAdd(V.spawn_ctr, (uint32_t)__popc(peers));
        if (mr) b_r = atomicAdd(V.spawn_ctr + 1, (uint32_t)__popc(mr));
        if (mt) b_t = atomicAdd(V.spawn_ctr + 2, (uint32_t)__popc(mt));
    }
    b_rec = __shfl_sync(peers, b_rec, leader); b_r = __shfl_sync(peers, b_r, leader); b_t = __shfl_sync(peers, b_t, leader);
    const unsigned below = (1u << lane) - 1u;
    if (has_r) {
        rec.child_r = b_r + __popc(mr & below);
        double* o = V.next_rays + 6 * (size_t)rec.child_r; o[0] = rr.o.x; o[1] = rr.o.y; o[2] = rr.o.z; o[3] = rr.d.x; o[4] = rr.d.y; o[5] = rr.d.z;
    }
    if (has_t) {
        rec.child_t = V.next_t_base + b_t + __popc(mt & below);
        double* o = V.next_rays + 6 * (size_t)rec.child_t; o[0] = rt.o.x; o[1] = rt.o.y; o[2] = rt.o.z; o[3] = rt.d.x; o[4] = rt.d.y; o[5] = rt.d.z;
    }
    V.recs[b_rec + __popc(peers & below)] = rec;
}

// GENERAL (scenes with Oren-Nayar, metal, glass or mirror; never FUSED): every material's BSDF::f, and the slots whose closest hit
// carries specular lobes are listed for k_secondary.
template <bool INST, bool FUSED, bool GENERAL = false, bool RAYBUF = false, bool LINEAR = false>
__global__ void __launch_bounds__(256, GENERAL ? LGB_GSHADE_MIN_BLOCKS : LGB_SHADE_MIN_BLOCKS) k_shade(DevScene S, DevCamera C, DevShade sh, DevWork W, DevOut O, DevWave V) {
    const double PI = 3.14159265358979323846264338327950288;
    const uint64_t total = W.n_pixels * W.spp;
    __shared__ double rad[FUSED ? 256 * 3 : 3];
    __shared__ unsigned char valid[FUSED ? 256 : 1];
    uint64_t g;
    bool mine;
    if (FUSED) {
        const uint32_t ppb = blockDim.x / W.spp;                        // pixels per block
        const uint64_t p = (uint64_t)blockIdx.x * ppb + threadIdx.x / W.spp;
        mine = threadIdx.x < ppb * W.spp && p < W.n_pixels;
        g = p * W.spp + threadIdx.x % W.spp;
    } else {
        g = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
        mine = g < total;
    }
    D3 output = d3(0, 0, 0);
    bool have = false;
    uint32_t x = 0, y = 0, s = 0;
    if (mine) {
        const uint32_t ref = V.hit_ref[g];
        Ray64 ray;
        if (ref != kSlotUnused && slot_ray<RAYBUF>(C, W, g, ray, x, y, s)) {
            have = true;
            if (ref == LGB_MISS) {                                       // background.rs:25-34
                output = background_of(sh, ray.d);
            } else {
                ShadePoint P; uint32_t id;
                shade_point<true, INST, GENERAL>(S, ray, V.hit_t[g], ref, P, id);
                const bool general = GENERAL && (P.B.flags & kMatGeneral);
                if (GENERAL && (P.B.flags & kMatSpecular) && W.depth < S.recursion && V.recs) spawn_children(P, V, (uint32_t)g);   // integrate.rs:69
                else if (GENERAL && (P.B.flags & kMatSpecular) && W.depth < S.recursion) {                                      // ... or k_secondary follows
                    const unsigned peers = __activemask();
                    const unsigned lane = threadIdx.x & 31u, leader = __ffs(peers) - 1;
                    uint32_t base = 0;
                    if (lane == leader) base = atomicAdd(V.sec_count, (uint32_t)__popc(peers));
                    base = __shfl_sync(peers, base, leader);
                    V.sec_list[base + __popc(peers & ((1u << lane) - 1u))] = (uint32_t)g;
                }
                const uint32_t occl = V.occl[g];
                if (O.aov_occl) O.aov_occl[((uint64_t)y * W.w + x) * W.spp + s] = occl;
                for (uint32_t l = 0; l < S.n_lights; l++) {              // integrate.rs:47-66
                    if ((occl >> l) & 1u) continue;
                    const double* L = S.lights + 9 * (size_t)l;
                    D3 wi = d3(L[0], L[1], L[2]) - P.ps;
                    double dist = sqrt(dot(wi, wi));
                    double f_att = L[6] + L[7] * dist + L[8] * dist * dist;
                    if (f_att == 0.0) continue;
                    wi = wi * (1.0 / dist);
                    double wi_dot_n = dot(wi, P.ns);
                    D3 f = general ? bsdf_f_general(P.B, wi) : bsdf_f(P.B, wi);     // zero when the shadow ray was skipped
                    output = output + mul_el(PI * d3(L[3], L[4], L[5]), f) * wi_dot_n / f_att;        // integrate.rs:65: (.. * wi_dot_n) / f_att
                }
                output = output + mul_el(d3(sh.ambient[0], sh.ambient[1], sh.ambient[2]), general ? bsdf_f_general(P.B, P.ns) : bsdf_f(P.B, P.ns));   // integrate.rs:67
                D3 zero = d3(0, 0, 0);
                output = output + zero + zero;          // integrate.rs:79 (reflected + refracted are zero for plastic)
            }
        }
    }
    if (!FUSED) {
        if (have) { O.radiance[3 * g + 0] = output.x; O.radiance[3 * g + 1] = output.y; O.radiance[3 * g + 2] = output.z; }
        return;
    }
    rad[3 * threadIdx.x] = output.x; rad[3 * threadIdx.x + 1] = output.y; rad[3 * threadIdx.x + 2] = output.z;
    valid[threadIdx.x] = have ? 1 : 0;
    __syncthreads();
    if (mine && threadIdx.x % W.spp == 0 && valid[threadIdx.x]) {        // sample 0 of a pixel inside the film: resolve it
        D3 c = d3(0, 0, 0);
        for (uint32_t k = 0; k < W.spp; k++) c = c + d3(rad[3 * (threadIdx.x + k)], rad[3 * (threadIdx.x + k) + 1], rad[3 * (threadIdx.x + k) + 2]);
        c = c * (1.0 / (double)W.spp);
        const uint64_t p = (uint32_t)g / W.spp;
        if constexpr (LINEAR) store_linear(O.film, W.compact_out ? W.compact_base + p : (uint64_t)y * W.w + x, c);
        else reinterpret_cast<uchar4*>(O.film)[W.compact_out ? W.compact_base + p : (uint64_t)y * W.w + x] = quantise(c);
    }
}

// ------------------------------------------------------------------ lean shading (plastic / matte(0) scenes without transformed aggregates)
// The same radiance as k_shade's plain variant, arranged for the FP64 pipe: the surface record comes from lean_surface + k_setup's
// sign byte; the shading frame never appears (the lobes are isotropic and (ss, ts, ns) is orthonormal, so wo_l.z = wo.ns,
// wi_l.z = wi.ns, wh = wi + wo with |wh|^2 = 2u, wi_l.wh = u, u = 1 + wi.wo); and all quotients of one BSDF evaluation share one
// reciprocal:
//   cos(theta_h)^2 = z^2 / 2u, z = wi.ns + wo.ns        q = alpha^2 c2 + s2 = Q / 2u, Q = alpha^2 z^2 + max(2u - z^2, 0)
//   Fresnel at cos = sqrt(u / 2) (fresnel.rs:37-64, eta 1 -> 1.5):  F = Fnum / Fden, Fnum = (ad)^2 + (cb)^2, Fden = 2 (bd)^2
//   4 cos_i cos_o (1 + Lambda_o + Lambda_i) = 2 (A_o cos_i + A_i cos_o), A(w) = sqrt(cos^2 + alpha^2 sin^2)   (microfacet.rs:55-66)
//   f_glossy wi.ns / f_att = ks alpha^2 Fnum (2u)^2 wi.ns / (pi Q^2 2 (A_o cos_i + A_i cos_o) Fden f_att)
// Four square roots and one reciprocal per evaluation, each a MUFU seed plus one refinement (lgb_math.cuh), against 9 IEEE
// divisions / square roots in bsdf_f.  The result differs from the reference's by f64 rounding, as bsdf_f's does.
struct LeanHit { D3 wo, ns; double woz, cos_o, Ao, alpha2; bool glossy; };
__device__ __forceinline__ void lean_eval(const LeanHit& H, D3 wi, double wn, double f_att, double& a, double& g) {
    const double PI = 3.14159265358979323846264338327950288;
    g = 0.0;
    const double cos_i = fabs(wn);
    if (H.glossy && cos_i != 0.0) {                                      // (cos_o != 0: the caller returns black for wo_l.z == 0)
        const double u = 1.0 + fdot(wi, H.wo);
        const double z = wn + H.woz, z2 = z * z;
        if (u > 0.0 && z2 != 0.0) {
            const double twou = u + u;
            const double Q = fma(H.alpha2, z2, fmax(twou - z2, 0.0));
            const double c = fmin(fast_sqrt(0.5 * u), 1.0);
            const double cos_t = fast_sqrt(fmax(fma(fma(c, c, -1.0), 4.0 / 9.0, 1.0), 0.0));    // 1 - (1 - c^2) / 1.5^2
            const double ta = fma(1.5, c, -cos_t), tb = fma(1.5, c, cos_t), tc = fma(-1.5, cos_t, c), td = fma(1.5, cos_t, c);
            const double ad = ta * td, cb = tc * tb, bd = tb * td;
            const double fnum = fma(ad, ad, cb * cb), fden = 2.0 * (bd * bd);
            const double Ai = fast_sqrt(fma(H.alpha2, fmax(fma(-cos_i, cos_i, 1.0), 0.0), cos_i * cos_i));
            const double K = PI * (Q * Q) * (2.0 * fma(H.Ao, cos_i, Ai * H.cos_o)) * fden;      // everything under the bar but f_att
            if (K > 0.0) {
                const double R = fast_rcp(K * f_att);
                g = H.alpha2 * fnum * (twou * twou) * R * wn;
                a = wn * K * R;
                return;
            }
        }
    }
    a = wn * fast_rcp(f_att);
}

// integrate.rs:47-67 for a plastic / matte(0) hit whose surface record is lean (lean_surface): `lit` = the lights that contribute.
__device__ __forceinline__ D3 lean_radiance(const DevScene& S, const DevShade& sh, const Ray64& ray, double t, const LeanSurf& Ls, uint32_t sflags, uint32_t lit) {
    const double PI = 3.14159265358979323846264338327950288;
    D3 output = d3(0, 0, 0);
    LeanHit H;
    H.ns = (sflags & kSfNsFlip) ? -Ls.n : Ls.n;
    const D3 ng = (sflags & kSfNgFlip) ? -Ls.n : Ls.n;
    const D3 ps = fmadd(ng, 2.220446049250313e-16 * 65536.0, fmadd(ray.d, t, ray.o));
    H.wo = ray.d * -fast_rsqrt(fdot(ray.d, ray.d));
    H.woz = fdot(H.wo, H.ns); H.cos_o = fabs(H.woz);
    const double* M = S.materials + kMatStride * (size_t)Ls.material;
    const uint32_t mflags = (uint32_t)__double_as_longlong(M[7]);
    H.glossy = mflags & kMatGlossy; H.alpha2 = M[3] * M[3];
    H.Ao = H.glossy ? fast_sqrt(fma(H.alpha2, fmax(fma(-H.cos_o, H.cos_o, 1.0), 0.0), H.cos_o * H.cos_o)) : 0.0;
    if (H.woz != 0.0) {                                  // bsdf.rs:82: every lobe is zero at wo_l.z == 0
        D3 dsum = d3(0, 0, 0), gsum = d3(0, 0, 0);       // sum of (pi I | ambient) x weight of the diffuse and of the glossy lobe
        for (uint32_t l = 0; l < S.n_lights; l++) {      // integrate.rs:47-66
            if (!((lit >> l) & 1u)) continue;
            const double* L = S.lights + 9 * (size_t)l;
            const D3 v = d3(L[0], L[1], L[2]) - ps;
            const double d2 = fdot(v, v);
            if (!(d2 > 0.0)) continue;
            const double inv = fast_rsqrt(d2), dist = d2 * inv;
            const double f_att = fma(L[8] * dist, dist, fma(L[7], dist, L[6]));
            if (f_att == 0.0) continue;
            const D3 wi = v * inv;
            double a, gl;
            lean_eval(H, wi, fdot(wi, H.ns), f_att, a, gl);
            const D3 I = PI * d3(L[3], L[4], L[5]);
            dsum = fmadd(I, a, dsum); gsum = fmadd(I, gl, gsum);
        }
        if (((sflags & kSfNsFlip) != 0) == ((sflags & kSfNgFlip) != 0)) {       // integrate.rs:67: wi = ns passes bsdf.rs:75 iff ns = ng
            double a, gl;
            lean_eval(H, H.ns, 1.0, 1.0, a, gl);
            const D3 amb = d3(sh.ambient[0], sh.ambient[1], sh.ambient[2]);
            dsum = fmadd(amb, a, dsum); gsum = fmadd(amb, gl, gsum);
        }
        const double inv_pi = 0.318309886183790671537767526745028724;
        const D3 kd = (mflags & kMatDiffuse) ? d3(M[0], M[1], M[2]) * inv_pi : d3(0, 0, 0);
        output = d3(fma(kd.x, dsum.x, M[4] * gsum.x), fma(kd.y, dsum.y, M[5] * gsum.y), fma(kd.z, dsum.z, M[6] * gsum.z));
    }
    return output;
}

// The slots lean_surface leaves to the reference's own sequence (vertex normals, sign decisions within rounding of a tie).
__device__ __forceinline__ D3 shade_generic_plastic(const DevScene& S, const DevShade& sh, const Ray64& ray, double t, uint32_t ref, uint32_t occl) {
    const double PI = 3.14159265358979323846264338327950288;
    ShadePoint P; uint32_t id;
    shade_point<true, false, false>(S, ray, t, ref, P, id);
    D3 output = d3(0, 0, 0);
    for (uint32_t l = 0; l < S.n_lights; l++) {              // integrate.rs:47-66
        if ((occl >> l) & 1u) continue;
        const double* L = S.lights + 9 * (size_t)l;
        D3 wi = d3(L[0], L[1], L[2]) - P.ps;
        const double dist = sqrt(dot(wi, wi));
        const double f_att = L[6] + L[7] * dist + L[8] * dist * dist;
        if (f_att == 0.0) continue;
        wi = wi * (1.0 / dist);
        const double wi_dot_n = dot(wi, P.ns);
        output = output + mul_el(PI * d3(L[3], L[4], L[5]), bsdf_f(P.B, wi)) * wi_dot_n / f_att;
    }
    return output + mul_el(d3(sh.ambient[0], sh.ambient[1], sh.ambient[2]), bsdf_f(P.B, P.ns));   // integrate.rs:67
}

#ifndef LGB_LEAN_MIN_BLOCKS
#define LGB_LEAN_MIN_BLOCKS 5            // (of 256 threads: 64 / 48 / 40 registers = 4 / 5 / 6: 3.88 / 3.65 / 3.75 ms on mixed4k)
#endif
// FUSED (spp <= 256): a block holds whole pixels (thread t: pixel t / spp of the block, sample t % spp); the samples meet in shared
// memory, one thread per (pixel, channel) sums them in sample order (integrate.rs:16-20) and quantises (img.rs:56-67), one thread per
// pixel stores the uchar4.  LINEAR (FUSED only): the thread that sums a (pixel, channel) stores its f32 to the linear film itself.
constexpr int kRadStride = 256 + 16 + 1;           // per channel; index t + t / 16 keeps the per-pixel runs on different banks
template <bool FUSED, bool LINEAR = false>
__global__ void __launch_bounds__(256, LGB_LEAN_MIN_BLOCKS) k_shade_lean(DevScene S, DevCamera C, DevShade sh, DevWork W, DevOut O, DevWave V) {
    const double PI = 3.14159265358979323846264338327950288;
    __shared__ double rad[FUSED ? 3 * kRadStride : 3];
    __shared__ unsigned char valid[FUSED ? 256 : 1];
    __shared__ unsigned char bytes[FUSED && !LINEAR ? 256 * 3 : 1];
    uint64_t g;
    uint32_t p32, s;
    bool mine;
    const uint32_t ppb = FUSED ? fdiv(blockDim.x, W.fd_spp) : 0u;   // pixels per block
    if constexpr (FUSED) {
        const uint32_t tp = fdiv(threadIdx.x, W.fd_spp);
        s = threadIdx.x - tp * W.spp;
        const uint64_t p = ((uint64_t)blockIdx.x + W.block_off) * ppb + tp;
        mine = tp < ppb && p < W.n_pixels;
        p32 = (uint32_t)p;
        g = p * W.spp + s;
    } else {
        g = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
        mine = g < W.n_pixels * W.spp;
        p32 = fdiv((uint32_t)g, W.fd_spp);
        s = (uint32_t)g - p32 * W.spp;
    }
    D3 output = d3(0, 0, 0);
    bool have = false, generic = false;
    uint32_t x = 0, y = 0;
    if (mine) {
        // everything the slot needs from the wave, requested at once (the loads are independent; their latency is this kernel's main stall)
        const uint32_t ref = wld(&V.hit_ref[g]);
        const double t = wld(&V.hit_t[g]);
        const uint32_t occl = wld(&V.occl[g]), gate = wld(&V.gate[g]), sflags = wld(&V.sflags[g]);
        if (ref != kSlotUnused && slot_to_pixel(W, p32, x, y)) {
            const Ray64 ray = camera_ray(C, W, x, y, s);
            have = true;
            if (ref == LGB_MISS) {                                       // background.rs:25-34
                output = background_of(sh, ray.d);
            } else {
                if (O.aov_occl) O.aov_occl[((uint64_t)y * W.w + x) * W.spp + s] = occl;
                if (sflags & kSfGeneric) generic = true;             // (rare: shaded after the lean code so that their registers do not add up)
                else {
                    LeanSurf Ls;
                    lean_surface<false>(S, ray, t, ref, sflags, Ls);
                    output = lean_radiance(S, sh, ray, t, Ls, sflags, gate & ~occl);      // lights neither occluded nor on the far side of ng
                }
            }
        }
    }
    if (generic) {
        const Ray64 ray = camera_ray(C, W, x, y, s);
        output = shade_generic_plastic(S, sh, ray, V.hit_t[g], V.hit_ref[g], V.occl[g]);
    }
    if constexpr (!FUSED) {
        if (have) { O.radiance[3 * g + 0] = output.x; O.radiance[3 * g + 1] = output.y; O.radiance[3 * g + 2] = output.z; }
    } else {
    {
        const uint32_t at = threadIdx.x + (threadIdx.x >> 4);
        rad[at] = output.x; rad[kRadStride + at] = output.y; rad[2 * kRadStride + at] = output.z;
        valid[threadIdx.x] = have ? 1 : 0;
    }
    __syncthreads();
    for (uint32_t j = threadIdx.x; j < 3u * ppb; j += blockDim.x) {        // item j: channel j / ppb of pixel j % ppb
        const uint32_t ch = j >= 2u * ppb ? 2u : (j >= ppb ? 1u : 0u), q = j - ch * ppb, t0 = q * W.spp;
        if (!valid[t0]) continue;
        const double* r = rad + ch * kRadStride;
        double c = 0.0;
        for (uint32_t k = 0; k < W.spp; k++) c = c + r[t0 + k + ((t0 + k) >> 4)];
        c = c * (1.0 / (double)W.spp);
        if constexpr (LINEAR) {
            const uint64_t p = ((uint64_t)blockIdx.x + W.block_off) * ppb + q;
            uint32_t px, py;
            slot_to_pixel(W, p, px, py);
            reinterpret_cast<float*>(O.film)[3 * (W.compact_out ? W.compact_base + p : (uint64_t)py * W.w + px) + ch] = __double2float_rn(c);
        } else {
            bytes[3 * q + ch] = (unsigned char)round(fmin(fmax(c, 0.0), 1.0) * 255.0);      // img.rs:56-67
        }
    }
    if constexpr (!LINEAR) {
    __syncthreads();
    if (threadIdx.x < ppb && valid[threadIdx.x * W.spp]) {
        const uint64_t p = ((uint64_t)blockIdx.x + W.block_off) * ppb + threadIdx.x;
        uint32_t px, py;
        slot_to_pixel(W, p, px, py);
        uchar4 o; o.x = bytes[3 * threadIdx.x]; o.y = bytes[3 * threadIdx.x + 1]; o.z = bytes[3 * threadIdx.x + 2]; o.w = 255;
        reinterpret_cast<uchar4*>(O.film)[W.compact_out ? W.compact_base + p : (uint64_t)py * W.w + px] = o;
    }
    }
    }
}

// Whitted recursion (integrate.rs:69-132) below the closest hits that carry specular lobes (glass, mirror), one thread per listed
// slot: a depth-first walk of the slot's ray tree on a per-thread stack of (ray, throughput, depth).  A node of the tree is shaded
// exactly as a primary hit is — closest hit, one shadow ray per light that can contribute, BSDF::f, ambient — and its radiance,
// scaled by the throughput of the path that reached it, is added to the slot's entry of the radiance buffer.
// The reference nests the products (spectrum x li(child)); the throughput form multiplies the same factors in another order, which
// moves the last bits of an f64 sum and nothing a byte of the film can see.
struct SecRay { Ray64 ray; D3 w; uint32_t depth; };
template <bool INST>
__device__ __forceinline__ void push_specular(const DevScene& S, const ShadePoint& P, D3 w, uint32_t depth, SecRay* stack, int& sp) {
    if (!(P.B.flags & kMatSpecular) || depth >= S.recursion) return;
    D3 spec, wi;
    if (sample_specular_reflection(P.B, spec, wi)) {                                  // specular_reflect, integrate.rs:82-106
        if (!(spec.x == 0.0 && spec.y == 0.0 && spec.z == 0.0) && !(dot(wi, P.ns) <= 0.0)) {
            SecRay& r = stack[sp++];
            r.ray.o = P.ps;
            r.ray.d = -1.0 * P.wo + 2.0 * dot(P.wo, P.ns) * P.ns;                     // bxdf::util::reflect, mod.rs:160-162
            r.w = mul_el(w, spec); r.depth = depth + 1;
        }
    }
    if (sample_specular_transmission(P.B, spec, wi)) {                                // specular_transmit, integrate.rs:108-132
        const double c = fabs(dot(wi, P.ns));
        if (!(spec.x == 0.0 && spec.y == 0.0 && spec.z == 0.0) && c != 0.0) {
            SecRay& r = stack[sp++];
            r.ray.o = P.pt; r.ray.d = wi;
            r.w = mul_el(w, spec) * c; r.depth = depth + 1;                             // pdf = 1
        }
    }
}
#ifndef LGB_SEC_THREADS
#define LGB_SEC_THREADS 128
#endif
#ifndef LGB_SEC_MIN_BLOCKS
#define LGB_SEC_MIN_BLOCKS 2
#endif
template <bool INST>
__global__ void __launch_bounds__(LGB_SEC_THREADS, LGB_SEC_MIN_BLOCKS) k_secondary(DevScene S, DevCamera C, DevShade sh, DevWork W, DevOut O, DevWave V) {
    const double PI = 3.14159265358979323846264338327950288;
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= *V.sec_count) return;
    const uint32_t g = V.sec_list[i];
    SecRay stack[kMaxRecursion + 1];
    int sp = 0;
    LocalCounters lc = {};
    unsigned long long traced = 0;
    {
        Ray64 ray; uint32_t x, y, s, id; ShadePoint P;
        slot_ray(C, W, g, ray, x, y, s);
        shade_point<true, INST, true>(S, ray, V.hit_t[g], V.hit_ref[g], P, id);
        push_specular<INST>(S, P, d3(1.0, 1.0, 1.0), 0, stack, sp);
    }
    D3 rad = d3(0, 0, 0);
    while (sp > 0) {
        const SecRay cur = stack[--sp];
        traced++;
        const Hit h = traverse<false, false, INST>(S, cur.ray, CUDART_INF, lc);
        if (h.ref == LGB_MISS) { rad = rad + mul_el(cur.w, background_of(sh, cur.ray.d)); continue; }
        ShadePoint P; uint32_t id;
        shade_point<true, INST, true>(S, cur.ray, h.t, h.ref, P, id);
        const bool general = P.B.flags & kMatGeneral;
        D3 output = d3(0, 0, 0);
        if (!(P.B.flags & kMatSpecular)) {                                  // specular lobes: BSDF::f is zero, no light can contribute
            for (uint32_t l = 0; l < S.n_lights; l++) {                      // integrate.rs:47-66
                const double* L = S.lights + 9 * (size_t)l;
                D3 wi = d3(L[0], L[1], L[2]) - P.ps;
                if (!(dot(wi, P.ng) * P.B.wo_ng > 0.0) || P.B.wo_l.z == 0.0) continue;     // every remaining lobe is REFLECTION: f = 0
                Ray64 sray; sray.o = P.ps; sray.d = wi;                      // light/point.rs:42-54: occluded iff the closest t < 1
                traced++;
                if (traverse<true, false, INST>(S, sray, 1.0, lc).ref != LGB_MISS) continue;
                const double dist = sqrt(dot(wi, wi));
                const double f_att = L[6] + L[7] * dist + L[8] * dist * dist;
                if (f_att == 0.0) continue;
                wi = wi * (1.0 / dist);
                const double wi_dot_n = dot(wi, P.ns);
                const D3 f = general ? bsdf_f_general(P.B, wi) : bsdf_f(P.B, wi);
                output = output + mul_el(PI * d3(L[3], L[4], L[5]), f) * wi_dot_n / f_att;        // integrate.rs:65: (.. * wi_dot_n) / f_att
            }
            output = output + mul_el(d3(sh.ambient[0], sh.ambient[1], sh.ambient[2]), general ? bsdf_f_general(P.B, P.ns) : bsdf_f(P.B, P.ns));
        }
        rad = rad + mul_el(cur.w, output);
        push_specular<INST>(S, P, cur.w, cur.depth, stack, sp);
    }
    O.radiance[3 * (size_t)g + 0] += rad.x; O.radiance[3 * (size_t)g + 1] += rad.y; O.radiance[3 * (size_t)g + 2] += rad.z;
    if (O.counters) atomicAdd(&ctr(O)->secondary_rays, traced);
}

// ---- the same recursion as a wavefront, one level of the ray trees at a time (the default; k_secondary is kept as a cross-check):
// the rays of a level are traced and shaded by the SAME lean kernels as the camera rays (k_primary / k_setup / k_shadow / k_shade
// in their RAYBUF variants: a slot's ray is read from a buffer instead of being generated by the camera), k_shade turns the specular
// hits of a level into the rays of the next one while it has their shading point in registers (spawn_children), and after the
// deepest level k_gather folds the radiance back up, parent by parent, in the reference's own order: output + reflected +
// refracted (integrate.rs:79).
__global__ void __launch_bounds__(256) k_gather(const SpawnRec* recs, const uint32_t* nspec, double* rad_parent, const double* rad_child) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= *nspec) return;
    const SpawnRec r = recs[i];
    D3 output = d3(rad_parent[3 * (size_t)r.slot], rad_parent[3 * (size_t)r.slot + 1], rad_parent[3 * (size_t)r.slot + 2]);
    D3 reflected = d3(0, 0, 0), refracted = d3(0, 0, 0);
    if (r.child_r != kNoChild) {
        const double* l = rad_child + 3 * (size_t)r.child_r;
        reflected = mul_el(d3(r.spec_r[0], r.spec_r[1], r.spec_r[2]), d3(l[0], l[1], l[2]));
    }
    if (r.child_t != kNoChild) {
        const double* l = rad_child + 3 * (size_t)r.child_t;
        refracted = mul_el(d3(r.spec_t[0], r.spec_t[1], r.spec_t[2]), d3(l[0], l[1], l[2])) * r.c;        // / pdf, which is 1
    }
    output = output + reflected + refracted;
    rad_parent[3 * (size_t)r.slot] = output.x; rad_parent[3 * (size_t)r.slot + 1] = output.y; rad_parent[3 * (size_t)r.slot + 2] = output.z;
}

// integrate.rs:16-20 + img.rs:56-67: in-order sum of the samples, weight, quantise, store.  LINEAR: the f32 store of store_linear instead.
template <bool LINEAR>
__global__ void __launch_bounds__(256) k_resolve(DevWork W, DevOut O) {
    const uint64_t p = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= W.n_pixels) return;
    uint32_t x, y;
    if (!slot_to_pixel(W, p, x, y)) return;
    const double weight = 1.0 / (double)W.spp;
    D3 c = d3(0, 0, 0);
    const double* r = O.radiance + 3 * p * W.spp;
    for (uint32_t s = 0; s < W.spp; s++) c = c + d3(r[3 * s], r[3 * s + 1], r[3 * s + 2]);
    c = c * weight;
    if constexpr (LINEAR) store_linear(O.film, W.compact_out ? W.compact_base + p : (uint64_t)y * W.w + x, c);
    else reinterpret_cast<uchar4*>(O.film)[W.compact_out ? W.compact_base + p : (uint64_t)y * W.w + x] = quantise(c);
}

// Per-sample radiance for lgb_capture_aov: radiance buffer (slot order) -> caller's order ((y * w + x) * spp + s).
__global__ void __launch_bounds__(256) k_export_li(DevWork W, DevOut O, DevWave V) {
    const uint64_t g = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= W.n_pixels * W.spp || V.hit_ref[g] == kSlotUnused) return;
    uint32_t x, y;
    const uint32_t p = fdiv((uint32_t)g, W.fd_spp), s = (uint32_t)g - p * W.spp;
    if (!slot_to_pixel(W, p, x, y)) return;
    const uint64_t gi = ((uint64_t)y * W.w + x) * W.spp + s;
    O.aov_li[3 * gi] = O.radiance[3 * g]; O.aov_li[3 * gi + 1] = O.radiance[3 * g + 1]; O.aov_li[3 * gi + 2] = O.radiance[3 * g + 2];
}

// Caller-supplied rays (lgb_trace_rays): closest hit id, t, RayIntersection::ng()/ns() (surface.rs:107-118)
// Parameter at which r enters B, or 0 if r starts inside B or misses it (f64 slab test; a zero direction component keeps its slab
// only if the origin lies in it).
__device__ __forceinline__ double entry_param(const TraceBox& B, const Ray64& r) {
    double tn = 0.0, tf = CUDART_INF;
#pragma unroll
    for (int k = 0; k < 3; k++) {
        const double o = comp(r.o, k), d = comp(r.d, k);
        if (d == 0.0) { if (o < B.lo[k] || o > B.hi[k]) return 0.0; continue; }
        const double t1 = (B.lo[k] - o) / d, t2 = (B.hi[k] - o) / d;
        tn = fmax(tn, fmin(t1, t2)); tf = fmin(tf, fmax(t1, t2));
    }
    return tn <= tf ? tn : 0.0;
}
// The world-space surface record of the closest hit `ref` on `ray` (formed in the primitive's own space, then brought back:
// bvh.rs:508-518), and its shading normal RayIntersection::ns() (surface.rs:107-118): lgb_trace_rays and lgb_capture_guides.
template <bool INST>
__device__ __forceinline__ void world_record(const DevScene& S, const Ray64& ray, uint32_t ref, double& t, Surf& sf) {
    if (INST) {
        const uint32_t space = space_of(S, ref);
        surface_of(S, ray_to_space(S, space, ray), ref, t, sf);
        record_to_world(S.spaces, space, sf);
    } else surface_of(S, ray, ref, t, sf);
}
__device__ __forceinline__ D3 shading_normal(const Surf& sf) { return sf.has_n ? normalize(sf.n) : normalize(cross(sf.s_dpdu, sf.s_dpdv)); }
template <bool INST>
__global__ void __launch_bounds__(128) k_trace(DevScene S, TraceBox B, const double* rays, uint64_t n, uint32_t* ids, double* ts, double* ngs, double* nss) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    Ray64 ray; ray.o = d3(rays[6 * i], rays[6 * i + 1], rays[6 * i + 2]); ray.d = d3(rays[6 * i + 3], rays[6 * i + 4], rays[6 * i + 5]);
    // The reference takes every ray through the root's Transform3, the identity included (bvh.rs:462): c0 x + c1 y + c2 z + c3 w
    // ends in + 0, which turns a -0 component into +0 (and so the octant, dinv = +inf, and the slab of an in-plane ray).
    if (!INST || (S.spaces[0].flags & kSpaceIdentity)) {
        ray.o = d3(__dadd_rn(ray.o.x, 0.0), __dadd_rn(ray.o.y, 0.0), __dadd_rn(ray.o.z, 0.0));
        ray.d = d3(__dadd_rn(ray.d.x, 0.0), __dadd_rn(ray.d.y, 0.0), __dadd_rn(ray.d.z, 0.0));
    }
    // |d| far from 1: the f32 ray cannot carry it (components overflow to inf, or several reciprocals clamp to the same 1e30), so
    // the ray is traced as (o, d 2^e) with max |d_k| 2^e in [1, 2).  Every exact test then returns t 2^-e bit for bit (each of
    // their operations scales exactly by a power of two, and |d| in 2^[-1022/2, 1023/2] keeps the reference's own products
    // normal), so t comes back exactly; the octant is unchanged.
    const double dm = fmax(fabs(ray.d.x), fmax(fabs(ray.d.y), fabs(ray.d.z)));
    const int e = (dm > 0.0 && (dm < 0x1p-40 || dm > 0x1p40)) ? -ilogb(dm) : 0;
    Ray64 rs = ray;
    if (e) rs.d = d3(ldexp(ray.d.x, e), ldexp(ray.d.y, e), ldexp(ray.d.z, e));
    // An origin outside the box of the scene and its camera (lgb_trace_rays admits it up to one box extent away): its f32
    // rounding could move the ray by more than the node padding and the filter bands allow (they are derived from that box), so
    // the f32 ray starts where the ray enters the box, grown by a margin.  The exact tests still see the ray as given.
    const double t0 = entry_param(B, rs);
    LocalCounters lc = {};
    Hit h = t0 > 0.0 ? traverse<false, false, INST, true>(S, rs, CUDART_INF, lc, t0) : traverse<false, false, INST>(S, rs, CUDART_INF, lc);
    if (e && h.ref != LGB_MISS) h.t = ldexp(h.t, e);
    uint32_t id = LGB_MISS; D3 ng = d3(0, 0, 0), ns = d3(0, 0, 0);
    if (h.ref != LGB_MISS) {
        Surf sf; double t = h.t;
        world_record<INST>(S, ray, h.ref, t, sf);
        id = sf.id;
        ng = normalize(cross(sf.g_dpdu, sf.g_dpdv));
        ns = shading_normal(sf);
    }
    if (ids) ids[i] = id;
    if (ts) ts[i] = h.ref != LGB_MISS ? h.t : CUDART_INF;
    if (ngs) { ngs[3 * i] = ng.x; ngs[3 * i + 1] = ng.y; ngs[3 * i + 2] = ng.z; }
    if (nss) { nss[3 * i] = ns.x; nss[3 * i + 1] = ns.y; nss[3 * i + 2] = ns.z; }
}

// lgb_capture_guides: per-pixel geometry of the camera rays' closest hits, read from the wave (hit_t / hit_ref) after the primary
// phase and before anything overwrites it.  A block holds whole pixels (kGuideThreads / spp of them; above kGuideThreads samples,
// one pixel in passes of kGuideThreads samples): each thread takes one sample slot, rebuilds its camera ray and derives the shading
// normal of its hit as lgb_trace_rays does; the normals meet in shared memory, one thread per pixel sums them in sample order
// (camera.rs:137-145), counts the hits and stores every requested output.  The anchor sample (camera.rs:143) gives depth and id.
constexpr uint32_t kGuideThreads = 256;
constexpr int kGuideStride = kGuideThreads + kGuideThreads / 16;      // per component; index t + t / 16 as in k_shade_lean
template <bool INST>
__global__ void __launch_bounds__(kGuideThreads) k_guides(DevScene S, DevCamera C, DevWork W, DevWave V, DevGuides G) {
    __shared__ double nrm[3 * kGuideStride];
    __shared__ unsigned char hit[kGuideThreads];
    const bool passes_of_one = W.spp > kGuideThreads;
    const uint32_t ppb = passes_of_one ? 1u : fdiv(kGuideThreads, W.fd_spp);          // pixels per block
    const uint32_t tp = passes_of_one ? 0u : fdiv(threadIdx.x, W.fd_spp);              // this thread's pixel in the block
    const uint64_t p = (uint64_t)blockIdx.x * ppb + tp;
    uint32_t x = 0, y = 0;
    const bool on_film = tp < ppb && p < W.n_pixels && slot_to_pixel(W, p, x, y);
    // the thread that reduces pixel threadIdx.x of the block
    const uint64_t rp = (uint64_t)blockIdx.x * ppb + threadIdx.x;
    uint32_t rx = 0, ry = 0;
    const bool reducer = threadIdx.x < ppb && rp < W.n_pixels && slot_to_pixel(W, rp, rx, ry);
    D3 sum = d3(0, 0, 0);
    uint32_t hits = 0;
    for (uint32_t s0 = 0; s0 < W.spp; s0 += passes_of_one ? kGuideThreads : W.spp) {
        const uint32_t s = passes_of_one ? s0 + threadIdx.x : threadIdx.x - tp * W.spp;
        D3 n = d3(0, 0, 0);
        bool h = false;
        if (on_film && s < W.spp) {
            const uint64_t g = p * W.spp + s;
            const uint32_t ref = V.hit_ref[g];
            if (ref != LGB_MISS && ref != kSlotUnused) {
                Surf sf; double t = V.hit_t[g];
                world_record<INST>(S, camera_ray(C, W, x, y, s), ref, t, sf);
                n = shading_normal(sf);
                h = true;
            }
        }
        const uint32_t at = threadIdx.x + (threadIdx.x >> 4);
        nrm[at] = n.x; nrm[kGuideStride + at] = n.y; nrm[2 * kGuideStride + at] = n.z;
        hit[threadIdx.x] = h ? 1 : 0;
        __syncthreads();
        if (reducer) {
            const uint32_t t0 = passes_of_one ? 0u : threadIdx.x * W.spp, cnt = passes_of_one ? min(kGuideThreads, W.spp - s0) : W.spp;
            for (uint32_t k = t0; k < t0 + cnt; k++) {
                const uint32_t i = k + (k >> 4);
                sum = sum + d3(nrm[i], nrm[kGuideStride + i], nrm[2 * kGuideStride + i]);
                hits += hit[k];
            }
        }
        __syncthreads();
    }
    if (!reducer) return;
    const uint64_t o = W.compact_out ? W.compact_base + rp : (uint64_t)ry * W.w + rx;
    if (G.normal) {
        const D3 c = sum * (1.0 / (double)W.spp);
        G.normal[3 * o] = __double2float_rn(c.x); G.normal[3 * o + 1] = __double2float_rn(c.y); G.normal[3 * o + 2] = __double2float_rn(c.z);
    }
    if (G.coverage) G.coverage[o] = __double2float_rn((double)hits / (double)W.spp);
    if (G.depth || G.prim_id) {
        const uint64_t ga = rp * W.spp + W.anchor;
        const uint32_t ref = V.hit_ref[ga];
        if (G.depth) G.depth[o] = ref == LGB_MISS ? CUDART_INF_F : __double2float_rn(__dmul_rn(V.hit_t[ga], G.view_len));
        if (G.prim_id) G.prim_id[o] = ref == LGB_MISS ? LGB_MISS : canonical_id(S, ref);
    }
}

// ------------------------------------------------------------------ end-of-frame flags of a shared film (multi-GPU, one process per GPU)
// The ranks' pixels reach rank 0's film as plain peer stores; what is left of the "gather" is knowing when they have all arrived.
// Each rank ends its frame by storing the frame number into its own word of rank 0's memory (behind a system-scope fence, so the
// pixel stores are visible first); rank 0 ends its frame by waiting for every word -- a microsecond-scale kernel each, no collective.
__global__ void k_flag_signal(volatile uint32_t* flag, uint32_t value) {
    __threadfence_system();
    *flag = value;
    __threadfence_system();
}
__global__ void k_flag_wait(const volatile uint32_t* flags, uint32_t first, uint32_t n, uint32_t stride_words, uint32_t value, uint32_t* timed_out) {
    const uint32_t i = first + threadIdx.x;
    if (threadIdx.x < n) {
        unsigned long long spins = 0;
        while ((int32_t)(flags[(size_t)i * stride_words] - value) < 0) {      // (wrap-safe: frame numbers only grow)
            if (++spins > (1ull << 31)) { if (timed_out) *timed_out = 1u; break; }      // a lost rank must not hang the GPU: give up after ~minutes
            __nanosleep(200);
        }
    }
    __threadfence_system();
}
constexpr unsigned kCtrWords = sizeof(DevCounters) / 8;
__global__ void __launch_bounds__(32 * kCtrWords) k_fold_counters(DevCounters* base) {      // one warp per counter word
    const unsigned word = threadIdx.x >> 5, lane = threadIdx.x & 31u;
    unsigned long long sum = 0;
    for (uint32_t k = 1 + lane; k <= kCtrStripes; k += 32) sum += reinterpret_cast<const unsigned long long*>(reinterpret_cast<const char*>(base) + (size_t)k * kCtrStride)[word];
    for (int d = 16; d > 0; d >>= 1) sum += __shfl_xor_sync(0xFFFFFFFFu, sum, d);
    if (lane == 0) reinterpret_cast<unsigned long long*>(base)[word] = sum;
}
cudaError_t launch_fold_counters(DevCounters* base, cudaStream_t stream) {
    if (!base) return cudaSuccess;
    k_fold_counters<<<1, 32 * kCtrWords, 0, stream>>>(base);
    return cudaGetLastError();
}
cudaError_t launch_flag_signal(void* flag, uint32_t value, cudaStream_t stream) {
    k_flag_signal<<<1, 1, 0, stream>>>((volatile uint32_t*)flag, value);
    return cudaGetLastError();
}
cudaError_t launch_flag_wait(const void* flags, uint32_t first, uint32_t n, uint32_t stride_bytes, uint32_t value, cudaStream_t stream) {
    if (n == 0) return cudaSuccess;
    k_flag_wait<<<1, 32 * ((n + 31) / 32), 0, stream>>>((const volatile uint32_t*)flags, first, n, stride_bytes / 4, value, nullptr);
    return cudaGetLastError();
}

// ------------------------------------------------------------------ ceilings for the roofline report
__global__ void k_l2_read(const float4* __restrict__ buf, uint64_t n_vec, int iters, float* sink) {
    float acc = 0.0f;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (int it = 0; it < iters; it++)
        for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_vec; i += stride) {
            float4 v = __ldcg(&buf[i]);
            acc += v.x + v.y + v.z + v.w;
        }
    if (acc == 123456.789f) *sink = acc;
}
__global__ void k_fp32_peak(int iters, float* sink) {
    float a0 = threadIdx.x * 1e-3f, a1 = a0 + 1.0f, a2 = a0 + 2.0f, a3 = a0 + 3.0f, a4 = a0 + 4.0f, a5 = a0 + 5.0f, a6 = a0 + 6.0f, a7 = a0 + 7.0f;
    const float m = 1.0000001f, c = 1e-7f;
    for (int i = 0; i < iters; i++) {
        a0 = __fmaf_rn(a0, m, c); a1 = __fmaf_rn(a1, m, c); a2 = __fmaf_rn(a2, m, c); a3 = __fmaf_rn(a3, m, c);
        a4 = __fmaf_rn(a4, m, c); a5 = __fmaf_rn(a5, m, c); a6 = __fmaf_rn(a6, m, c); a7 = __fmaf_rn(a7, m, c);
    }
    float s = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
    if (s == 123456.789f) *sink = s;
}
__global__ void k_fp64_peak(int iters, double* sink) {
    double a0 = threadIdx.x * 1e-3, a1 = a0 + 1.0, a2 = a0 + 2.0, a3 = a0 + 3.0, a4 = a0 + 4.0, a5 = a0 + 5.0, a6 = a0 + 6.0, a7 = a0 + 7.0;
    const double m = 1.0000001, c = 1e-7;
    for (int i = 0; i < iters; i++) {
        a0 = __fma_rn(a0, m, c); a1 = __fma_rn(a1, m, c); a2 = __fma_rn(a2, m, c); a3 = __fma_rn(a3, m, c);
        a4 = __fma_rn(a4, m, c); a5 = __fma_rn(a5, m, c); a6 = __fma_rn(a6, m, c); a7 = __fma_rn(a7, m, c);
    }
    double s = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
    if (s == 123456.789) *sink = s;
}

// The shading path's reciprocal / reciprocal square root (lgb_math.cuh) on caller-supplied values: tests pin their accuracy.
__global__ void k_fastmath(const double* x, uint64_t n, double* rcp, double* rsq) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) { rcp[i] = fast_rcp(x[i]); rsq[i] = fast_rsqrt(x[i]); }
}
cudaError_t launch_fastmath(const double* x, uint64_t n, double* rcp, double* rsq, cudaStream_t stream) {
    if (n) k_fastmath<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(x, n, rcp, rsq);
    return cudaGetLastError();
}

// ------------------------------------------------------------------ launch wrappers (called from lgb_api.cu)
bool render_fused(uint32_t spp) { return spp >= 1 && spp <= 256; }      // and !S.general: see launch_render

// `ev` (optional): kRenderEvents events recorded around the phases: start | primary | setup | anchor shadow rays |
// pretest + remaining shadow rays | shade | resolve.
// part 1 = k_primary (every slot, or W.slot_list: the re-trace of tied slots), 2 = everything after it, 3 = both.
// `guides` (optional, part 2): k_guides first, in the primary phase of `ev`; with O.film == NULL the frame ends there (a geometry pass).
// `side` (optional): the shadow chains of the lights are independent of each other (own queues, own fetch counters, own occluder
// table, one bit each in `occl`), so they are dealt round-robin over the launch stream and the side streams: the blocks of one
// light's persistent kernel fill the SMs that the tail of another's has left idle.
#define KL(nm, light, st, ...) do { if (klog) klog->begin(nm, light, st); __VA_ARGS__; if (klog) klog->end(st, O.counters); } while (0)
cudaError_t launch_render(const DevScene& S, const DevCamera& C, const DevShade& sh, const DevWork& W, const DevOut& O,
                          const DevWave& V, bool stats, bool all_shadows, int sms, cudaStream_t stream, cudaEvent_t* ev, int part, const SideStreams* side,
                          KernelLog* klog, ShadeChunks* chunks, bool linear, const DevGuides* guides) {
    if (chunks) chunks->launched = 0;
    auto mark = [&](int i) { if (ev) cudaEventRecord(ev[i], stream); };
    const uint64_t total = W.n_pixels * W.spp;
    const bool cache = W.spp > 1;
    const unsigned pblocks = (unsigned)std::min<uint64_t>((total + LGB_TRAV_THREADS - 1) / LGB_TRAV_THREADS, (uint64_t)sms * LGB_MIN_BLOCKS);
    const bool inst = S.instanced != 0;      // transformed aggregates: the INST kernel variants (the plain ones carry no trace of them)
    cudaError_t e;
    if (part & 1) {
        if (!W.slot_list) mark(0);
        if (total == 0) return cudaSuccess;
        if (!W.slot_list) {
            if ((e = cudaMemsetAsync(V.work_counter, 0, kWaveCtrBytes, stream)) != cudaSuccess) return e;
            if (cache && S.n_lights && !(S.grids && !inst) && (e = cudaMemsetAsync(V.occluder, 0xFF, (size_t)S.n_lights * W.n_pixels * 4, stream)) != cudaSuccess) return e;      // (light grids keep no occluder cache)
        } else if ((e = cudaMemsetAsync(V.work_counter, 0, 8, stream)) != cudaSuccess) return e;      // the fetch counter restarts for the listed slots
        const uint64_t work = W.slot_list ? W.n_list : total;
        const unsigned pb = (unsigned)std::min<uint64_t>((work + LGB_TRAV_THREADS - 1) / LGB_TRAV_THREADS, (uint64_t)sms * LGB_MIN_BLOCKS);
        if (W.cg_start && !inst && !W.slot_list) {
            const unsigned cb = (unsigned)((total + LGB_CPRIMARY_THREADS - 1) / LGB_CPRIMARY_THREADS);
            if (W.setup_in_primary) KL("k_cprimary(+setup)", -1, stream, if (stats) k_cprimary<true, true><<<cb, LGB_CPRIMARY_THREADS, 0, stream>>>(S, C, W, O, V); else k_cprimary<false, true><<<cb, LGB_CPRIMARY_THREADS, 0, stream>>>(S, C, W, O, V));
            else KL("k_cprimary", -1, stream, if (stats) k_cprimary<true><<<cb, LGB_CPRIMARY_THREADS, 0, stream>>>(S, C, W, O, V); else k_cprimary<false><<<cb, LGB_CPRIMARY_THREADS, 0, stream>>>(S, C, W, O, V));
        } else if (W.beams && W.spp >= 4 && !inst && !W.slot_list) {
            // one bundle traversal per pixel, then every sample ray walks its pixel's leaf list; pixels whose bundle
            // reaches too many leaves go through the per-ray traversal (their slots are listed by k_leafp)
            const unsigned bb = (unsigned)((W.n_pixels + LGB_BEAM_THREADS - 1) / LGB_BEAM_THREADS), lb = (unsigned)((total + LGB_LEAFP_THREADS - 1) / LGB_LEAFP_THREADS);
            KL("k_beam", -1, stream, if (stats) k_beam<true><<<bb, LGB_BEAM_THREADS, 0, stream>>>(S, C, W, O, V); else k_beam<false><<<bb, LGB_BEAM_THREADS, 0, stream>>>(S, C, W, O, V));
            KL("k_leafp", -1, stream, if (stats) k_leafp<true><<<lb, LGB_LEAFP_THREADS, 0, stream>>>(S, C, W, O, V); else k_leafp<false><<<lb, LGB_LEAFP_THREADS, 0, stream>>>(S, C, W, O, V));
            DevWork Wf = W; Wf.slot_list = V.fallback_list; Wf.n_list = 0; Wf.n_list_dev = V.fallback_count;
            KL("k_primary(fallback)", -1, stream, if (stats) k_primary<true, false><<<pb, LGB_TRAV_THREADS, 0, stream>>>(S, C, Wf, O, V); else k_primary<false, false><<<pb, LGB_TRAV_THREADS, 0, stream>>>(S, C, Wf, O, V));
        } else if (pb) {
            if (inst) KL("k_primary", -1, stream, if (stats) k_primary<true, true><<<pb, LGB_TRAV_THREADS, 0, stream>>>(S, C, W, O, V); else k_primary<false, true><<<pb, LGB_TRAV_THREADS, 0, stream>>>(S, C, W, O, V));
            else KL("k_primary", -1, stream, if (stats) k_primary<true, false><<<pb, LGB_TRAV_THREADS, 0, stream>>>(S, C, W, O, V); else k_primary<false, false><<<pb, LGB_TRAV_THREADS, 0, stream>>>(S, C, W, O, V));
        }
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
    }
    if (!(part & 2)) return cudaSuccess;
    if (total == 0) return cudaSuccess;
    if (guides) {                       // every slot's final hit is in the wave (the tie re-trace, if any, is done); nothing has overwritten it yet
        const unsigned gppb = W.spp <= kGuideThreads ? kGuideThreads / W.spp : 1u, gb = (unsigned)((W.n_pixels + gppb - 1) / gppb);
        KL("k_guides", -1, stream, if (inst) k_guides<true><<<gb, kGuideThreads, 0, stream>>>(S, C, W, V, *guides); else k_guides<false><<<gb, kGuideThreads, 0, stream>>>(S, C, W, V, *guides));
        if (!O.film) {                  // a geometry pass: no setup, shadow, shade or resolve work
            for (int k = 1; k <= 6; k++) mark(k);
            return cudaGetLastError();
        }
    }
    mark(1);
    const unsigned blocks = (unsigned)((total + 255) / 256), ablocks = (unsigned)((total + kAppendThreads - 1) / kAppendThreads);
    if (W.setup_in_primary) {           // k_cprimary<SETUP> has written ps / gate / sign byte: straight to the shadow rays
        mark(2);
        KL("k_gshadow", -1, stream, if (stats) k_gshadow<true, false><<<(unsigned)((total + LGB_GSHADOW_THREADS - 1) / LGB_GSHADOW_THREADS), LGB_GSHADOW_THREADS, 0, stream>>>(S, C, W, O, V); else k_gshadow<false, false><<<(unsigned)((total + LGB_GSHADOW_THREADS - 1) / LGB_GSHADOW_THREADS), LGB_GSHADOW_THREADS, 0, stream>>>(S, C, W, O, V));
        mark(3);
    } else {
    if (inst) KL("k_setup", -1, stream, if (all_shadows) k_setup<true, true><<<ablocks, kAppendThreads, 0, stream>>>(S, C, sh, W, O, V); else k_setup<false, true><<<ablocks, kAppendThreads, 0, stream>>>(S, C, sh, W, O, V));
    else KL("k_setup", -1, stream, if (all_shadows) k_setup<true, false><<<ablocks, kAppendThreads, 0, stream>>>(S, C, sh, W, O, V); else k_setup<false, false><<<ablocks, kAppendThreads, 0, stream>>>(S, C, sh, W, O, V));
    mark(2);
    if (S.grids && !inst) {             // light grids: every shadow ray of the frame in one launch, no traversal (lgb_grid.cu)
        if (stats) KL("k_gshadow", -1, stream, if (all_shadows) k_gshadow<true, true><<<(unsigned)((total + LGB_GSHADOW_THREADS - 1) / LGB_GSHADOW_THREADS), LGB_GSHADOW_THREADS, 0, stream>>>(S, C, W, O, V); else k_gshadow<true, false><<<(unsigned)((total + LGB_GSHADOW_THREADS - 1) / LGB_GSHADOW_THREADS), LGB_GSHADOW_THREADS, 0, stream>>>(S, C, W, O, V));
        else KL("k_gshadow", -1, stream, if (all_shadows) k_gshadow<false, true><<<(unsigned)((total + LGB_GSHADOW_THREADS - 1) / LGB_GSHADOW_THREADS), LGB_GSHADOW_THREADS, 0, stream>>>(S, C, W, O, V); else k_gshadow<false, false><<<(unsigned)((total + LGB_GSHADOW_THREADS - 1) / LGB_GSHADOW_THREADS), LGB_GSHADOW_THREADS, 0, stream>>>(S, C, W, O, V));
        mark(3);
    }
    }
    // per light: anchor rays (queue A), then the cached-occluder test of the rest (B -> C), then the survivors (queue C)
    const int nside = (side && S.n_lights > 1 && !S.grids) ? std::min<int>(side->n, (int)S.n_lights - 1) : 0;
    for (int k = 0; k < nside; k++) { cudaEventRecord(side->fork, stream); cudaStreamWaitEvent(side->s[k], side->fork, 0); }
    // (light by light on its lane: the shadow-beam lists of a lane are reused by its next light)
    for (uint32_t l = 0; l < (S.grids && !inst ? 0u : S.n_lights); l++) {
        const int lane = nside ? (int)(l % (uint32_t)(nside + 1)) : 0;
        cudaStream_t ls = lane ? side->s[lane - 1] : stream;
        uint2* blist = lane ? V.beam_list2 : V.beam_list; uint32_t* bcount = lane ? V.beam_count2 : V.beam_count;
        const bool sbeams = W.beams && cache && !inst && blist && lane < 2;
        for (int which = kQueueA; which <= (cache ? kQueueC : kQueueA); which += 2) {
            const unsigned sb = which == kQueueA ? (unsigned)std::min<uint64_t>((W.n_pixels + LGB_TRAV_THREADS - 1) / LGB_TRAV_THREADS, pblocks) : pblocks;
            if (which == kQueueC) {
                if (sbeams) {                       // pixels whose anchor ray is free: one bundle walk, then the other samples from its list, no traversal
                    if ((e = cudaMemsetAsync(bcount, 0xFF, (size_t)W.n_pixels * 4, ls)) != cudaSuccess) return e;
                    const unsigned bb = (unsigned)((W.n_pixels + LGB_SBEAM_THREADS_ - 1) / LGB_SBEAM_THREADS_);
                    KL("k_sbeam", (int)l, ls, if (stats) k_sbeam<true><<<bb, LGB_SBEAM_THREADS_, 0, ls>>>(S, W, O, V, l, blist, bcount); else k_sbeam<false><<<bb, LGB_SBEAM_THREADS_, 0, ls>>>(S, W, O, V, l, blist, bcount));
                    const unsigned wb = (unsigned)((total + LGB_SWALK_THREADS - 1) / LGB_SWALK_THREADS);
                    KL("k_swalk", (int)l, ls, if (stats) k_swalk<true><<<wb, LGB_SWALK_THREADS, 0, ls>>>(S, W, O, V, l, blist, bcount); else k_swalk<false><<<wb, LGB_SWALK_THREADS, 0, ls>>>(S, W, O, V, l, blist, bcount));
                }
                const unsigned tb = (unsigned)std::min<uint64_t>(ablocks, (uint64_t)sms * 4);
                KL("k_pretest", (int)l, ls, if (inst) k_pretest<true><<<tb, kAppendThreads, 0, ls>>>(S, W, O, V, l); else k_pretest<false><<<tb, kAppendThreads, 0, ls>>>(S, W, O, V, l));
            }
            const char* sname = which == kQueueA ? "k_shadow(anchors)" : "k_shadow(rest)";
            if (inst) KL(sname, (int)l, ls, if (stats) k_shadow<true, true><<<sb, LGB_TRAV_THREADS, 0, ls>>>(S, W, O, V, l, which); else k_shadow<false, true><<<sb, LGB_TRAV_THREADS, 0, ls>>>(S, W, O, V, l, which));
            else KL(sname, (int)l, ls, if (stats) k_shadow<true, false><<<sb, LGB_TRAV_THREADS, 0, ls>>>(S, W, O, V, l, which); else k_shadow<false, false><<<sb, LGB_TRAV_THREADS, 0, ls>>>(S, W, O, V, l, which));
            if (which == kQueueA && l == 0) mark(3);      // (the anchor / rest split of the first light only)
        }
    }
    if (S.n_lights == 0) mark(3);
    for (int k = 0; k < nside; k++) { cudaEventRecord(side->join[k], side->s[k]); cudaStreamWaitEvent(stream, side->join[k], 0); }
    mark(4);
    if (S.general) {                    // materials beyond plastic: every BSDF in k_shade, then the specular ray trees, then the film
        KL("k_shade(general)", -1, stream, if (inst) k_shade<true, false, true><<<blocks, 256, 0, stream>>>(S, C, sh, W, O, V); else k_shade<false, false, true><<<blocks, 256, 0, stream>>>(S, C, sh, W, O, V));
        if (part & 4) return cudaGetLastError();      // the caller runs the levels of the ray trees (launch_level / launch_spawn / launch_gather) and the resolve
        if (S.specular && S.recursion > 0) {
            const unsigned sb = (unsigned)((total + LGB_SEC_THREADS - 1) / LGB_SEC_THREADS);
            KL("k_secondary", -1, stream, if (inst) k_secondary<true><<<sb, LGB_SEC_THREADS, 0, stream>>>(S, C, sh, W, O, V); else k_secondary<false><<<sb, LGB_SEC_THREADS, 0, stream>>>(S, C, sh, W, O, V));
        }
        mark(5);
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
        KL("k_resolve", -1, stream, if (linear) k_resolve<true><<<(unsigned)((W.n_pixels + 255) / 256), 256, 0, stream>>>(W, O); else k_resolve<false><<<(unsigned)((W.n_pixels + 255) / 256), 256, 0, stream>>>(W, O));
    } else if (render_fused(W.spp) && !O.aov_li) {   // whole pixels per block: shade and resolve in one kernel, no radiance buffer
        const unsigned ft = W.spp <= LGB_FUSED_THREADS ? LGB_FUSED_THREADS : 256u;        // threads per block: whole pixels, as few of them as the option allows
        const unsigned fb = (unsigned)((W.n_pixels + (ft / W.spp) - 1) / (ft / W.spp));
        if (chunks && chunks->want > 1 && !inst && !klog && !linear && fb >= 64u * chunks->want) {      // (the RGBA8 read-back of lgb_capture)
            // slices of consecutive blocks = consecutive pixel slots = (single-rank tile lists are row-major) consecutive rows of macro tiles
            const unsigned K = std::min<unsigned>(chunks->want, 8u), ppb = ft / W.spp;
            for (unsigned k = 0; k < K; k++) {
                const unsigned b0 = (unsigned)((uint64_t)fb * k / K), b1 = (unsigned)((uint64_t)fb * (k + 1) / K);
                DevWork Wk = W; Wk.block_off = b0;
                k_shade_lean<true><<<b1 - b0, ft, 0, stream>>>(S, C, sh, Wk, O, V);
                cudaEventRecord(chunks->ev[k], stream);
                chunks->done_pixels[k] = std::min<uint64_t>((uint64_t)b1 * ppb, W.n_pixels);
            }
            chunks->launched = K;
        } else if (linear)
        KL(inst ? "k_shade(+linear film)" : "k_shade_lean(+linear film)", -1, stream, if (inst) k_shade<true, true, false, false, true><<<fb, ft, 0, stream>>>(S, C, sh, W, O, V); else k_shade_lean<true, true><<<fb, ft, 0, stream>>>(S, C, sh, W, O, V));
        else
        KL(inst ? "k_shade(+film)" : "k_shade_lean(+film)", -1, stream, if (inst) k_shade<true, true><<<fb, ft, 0, stream>>>(S, C, sh, W, O, V); else k_shade_lean<true><<<fb, ft, 0, stream>>>(S, C, sh, W, O, V));
        mark(5);
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
    } else {
        KL(inst ? "k_shade" : "k_shade_lean", -1, stream, if (inst) k_shade<true, false><<<blocks, 256, 0, stream>>>(S, C, sh, W, O, V); else k_shade_lean<false><<<blocks, 256, 0, stream>>>(S, C, sh, W, O, V));
        mark(5);
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
        KL("k_resolve", -1, stream, if (linear) k_resolve<true><<<(unsigned)((W.n_pixels + 255) / 256), 256, 0, stream>>>(W, O); else k_resolve<false><<<(unsigned)((W.n_pixels + 255) / 256), 256, 0, stream>>>(W, O));
    }
    mark(6);
    return cudaGetLastError();
}
#undef KL
// One level of the specular ray trees: W.mode == 3, the rays in W.rays; radiance of every ray into O.radiance, specular hits into V.sec_list.
cudaError_t launch_level(const DevScene& S, const DevCamera& C, const DevShade& sh, const DevWork& W, const DevOut& O, const DevWave& V, int sms, cudaStream_t stream, DevCounters* shadow_counters) {
    const uint64_t total = W.n_pixels;
    if (total == 0) return cudaSuccess;
    cudaError_t e;
    if ((e = cudaMemsetAsync(V.work_counter, 0, kWaveCtrBytes, stream)) != cudaSuccess) return e;
    const unsigned pb = (unsigned)std::min<uint64_t>((total + LGB_TRAV_THREADS - 1) / LGB_TRAV_THREADS, (uint64_t)sms * LGB_MIN_BLOCKS);
    const unsigned blocks = (unsigned)((total + 255) / 256), ablocks = (unsigned)((total + kAppendThreads - 1) / kAppendThreads);
    if (S.instanced) {
        k_primary<false, true, true><<<pb, LGB_TRAV_THREADS, 0, stream>>>(S, C, W, O, V);
        k_setup<false, true, true><<<ablocks, kAppendThreads, 0, stream>>>(S, C, sh, W, O, V);
        for (uint32_t l = 0; l < S.n_lights; l++) k_shadow<false, true><<<pb, LGB_TRAV_THREADS, 0, stream>>>(S, W, O, V, l, kQueueA);
        k_shade<true, false, true, true><<<blocks, 256, 0, stream>>>(S, C, sh, W, O, V);
    } else {
        k_primary<false, false, true><<<pb, LGB_TRAV_THREADS, 0, stream>>>(S, C, W, O, V);
        k_setup<false, false, true><<<ablocks, kAppendThreads, 0, stream>>>(S, C, sh, W, O, V);
        if (S.grids) { DevOut Os = O; Os.counters = shadow_counters; k_gshadow<false, false><<<(unsigned)((total + LGB_GSHADOW_THREADS - 1) / LGB_GSHADOW_THREADS), LGB_GSHADOW_THREADS, 0, stream>>>(S, C, W, Os, V); }
        else for (uint32_t l = 0; l < S.n_lights; l++) k_shadow<false, false><<<pb, LGB_TRAV_THREADS, 0, stream>>>(S, W, O, V, l, kQueueA);
        k_shade<false, false, true, true><<<blocks, 256, 0, stream>>>(S, C, sh, W, O, V);
    }
    return cudaGetLastError();
}
cudaError_t launch_gather(const SpawnRec* recs, const uint32_t* nspec, double* rad_parent, const double* rad_child, uint64_t n_upper, cudaStream_t stream) {
    if (n_upper == 0) return cudaSuccess;
    k_gather<<<(unsigned)((n_upper + 255) / 256), 256, 0, stream>>>(recs, nspec, rad_parent, rad_child);
    return cudaGetLastError();
}
cudaError_t launch_export_li(const DevWork& W, const DevOut& O, const DevWave& V, cudaStream_t stream) {
    const uint64_t total = W.n_pixels * W.spp;
    if (total == 0) return cudaSuccess;
    k_export_li<<<(unsigned)((total + 255) / 256), 256, 0, stream>>>(W, O, V);
    return cudaGetLastError();
}
cudaError_t launch_resolve(const DevWork& W, const DevOut& O, cudaStream_t stream, bool linear) {
    if (W.n_pixels == 0) return cudaSuccess;
    if (linear) k_resolve<true><<<(unsigned)((W.n_pixels + 255) / 256), 256, 0, stream>>>(W, O);
    else k_resolve<false><<<(unsigned)((W.n_pixels + 255) / 256), 256, 0, stream>>>(W, O);
    return cudaGetLastError();
}
cudaError_t launch_trace(const DevScene& S, const TraceBox& B, const double* rays, uint64_t n, uint32_t* ids, double* ts, double* ng, double* ns, cudaStream_t stream) {
    if (n == 0) return cudaSuccess;
    if (S.instanced) k_trace<true><<<(unsigned)((n + 127) / 128), 128, 0, stream>>>(S, B, rays, n, ids, ts, ng, ns);
    else k_trace<false><<<(unsigned)((n + 127) / 128), 128, 0, stream>>>(S, B, rays, n, ids, ts, ng, ns);
    return cudaGetLastError();
}
cudaError_t launch_l2_read(const void* buf, uint64_t bytes, int iters, float* sink, int sms, cudaStream_t stream) {
    k_l2_read<<<sms * 8, 256, 0, stream>>>(reinterpret_cast<const float4*>(buf), bytes / 16, iters, sink);
    return cudaGetLastError();
}
cudaError_t launch_fp32_peak(int iters, float* sink, int sms, cudaStream_t stream) {
    k_fp32_peak<<<sms * 8, 256, 0, stream>>>(iters, sink);
    return cudaGetLastError();
}
cudaError_t launch_fp64_peak(int iters, double* sink, int sms, cudaStream_t stream) {
    k_fp64_peak<<<sms * 8, 256, 0, stream>>>(iters, sink);
    return cudaGetLastError();
}

}  // namespace lgb
