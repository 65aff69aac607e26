// lasgun_oracle.cpp — TEST INFRASTRUCTURE ONLY.
//
// CPU f64 restatement of nfrasser/lasgun's per-pixel render loop, written from
// the reference's Rust sources (cited per function as file:line relative to
// /root/reference).  It is the checker for the CUDA path and the CPU baseline
// of bench.py; nothing under lasgun_b200/ may include, link or call it.
//
// Parity pin status: the sphere / cuboid / triangle / surface-interaction
// routines are pinned by the reference's own 16 unit-test vectors
// (tests/test_oracle_known_answers.py).  BVH build, traversal, camera,
// shading, shadows and film quantisation have NO reference test or golden
// image ("parity unpinned" for those rows); the Rust toolchain is absent here
// so the reference cannot be run.  They were restated line by line.
//
// Arithmetic rules: every operation is a plain IEEE-754 binary64 op in the
// reference's source order; build with -ffp-contract=off (no FMA fusion), no
// fast-math.  cgmath 0.17 semantics assumed (source not vendored):
//   dot = (x*x' + y*y') + z*z';  cross = (y z' - z y', z x' - x z', x y' - y x');
//   normalize(v) = v * (1 / sqrt(dot(v,v)));  vector/scalar divides per lane;
//   Matrix4 * Vector4 = c0*x + c1*y + c2*z + c3*w;  transform_point divides by w
//   via multiplication with (1/w).
// Rust semantics mirrored: f64::min/max ignore a NaN operand; `as u32` saturates
// and maps NaN to 0; f64::round is half-away-from-zero; signum(+0.0) = +1.

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <limits>
#include <memory>
#include <thread>
#include <vector>

namespace orc {

static const double PI = 3.14159265358979323846264338327950288;   // std::f64::consts::PI
static const double FRAC_1_PI = 0.318309886183790671537767526745028724;
static const double F64_MAX = std::numeric_limits<double>::max();
static const double INF = std::numeric_limits<double>::infinity();

// ---------------------------------------------------------------- vectors
struct V3 {
    double x, y, z;
    double operator[](int i) const { return i == 0 ? x : (i == 1 ? y : z); }
    double& at(int i) { return i == 0 ? x : (i == 1 ? y : z); }
};
static inline V3 v3(double x, double y, double z) { return V3{x, y, z}; }
static inline V3 operator+(V3 a, V3 b) { return v3(a.x + b.x, a.y + b.y, a.z + b.z); }
static inline V3 operator-(V3 a, V3 b) { return v3(a.x - b.x, a.y - b.y, a.z - b.z); }
static inline V3 operator-(V3 a) { return v3(-a.x, -a.y, -a.z); }
static inline V3 operator*(V3 a, double s) { return v3(a.x * s, a.y * s, a.z * s); }
static inline V3 operator*(double s, V3 a) { return v3(s * a.x, s * a.y, s * a.z); }
static inline V3 operator/(V3 a, double s) { return v3(a.x / s, a.y / s, a.z / s); }
static inline V3 mul_el(V3 a, V3 b) { return v3(a.x * b.x, a.y * b.y, a.z * b.z); }
static inline double dot(V3 a, V3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
static inline V3 cross(V3 a, V3 b) {
    return v3(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x);
}
static inline double magnitude(V3 a) { return std::sqrt(dot(a, a)); }
static inline V3 normalize(V3 a) { return a * (1.0 / magnitude(a)); }
static inline bool eq(V3 a, V3 b) { return a.x == b.x && a.y == b.y && a.z == b.z; }

// Rust f64::min / f64::max: if one operand is NaN the other is returned.
static inline double rmin(double a, double b) { return std::fmin(a, b); }
static inline double rmax(double a, double b) { return std::fmax(a, b); }
// space/bounds.rs:171-178 — generic min/max used by Bounds3 (plain `<`).
static inline double bmin(double a, double b) { return a < b ? a : b; }
static inline double bmax(double a, double b) { return a < b ? b : a; }
// Rust `f64 as u32`: saturating, NaN -> 0.
static inline uint32_t as_u32(double v) {
    if (!(v == v)) return 0;
    if (v <= 0.0) return 0;
    if (v >= 4294967295.0) return 4294967295u;
    return (uint32_t)v;
}

// ---------------------------------------------------------------- 4x4 (column major, cgmath)
struct M4 { double c[4][4]; };  // c[col][row]
static M4 m4_identity() {
    M4 m; std::memset(&m, 0, sizeof m);
    for (int i = 0; i < 4; i++) m.c[i][i] = 1.0;
    return m;
}
// cgmath Matrix4 * Matrix4: result column j = lhs * rhs.column(j).
static inline void m4_mulv(const M4& m, const double v[4], double out[4]) {
    for (int r = 0; r < 4; r++)
        out[r] = m.c[0][r] * v[0] + m.c[1][r] * v[1] + m.c[2][r] * v[2] + m.c[3][r] * v[3];
}
static M4 m4_mul(const M4& a, const M4& b) {
    M4 o;
    for (int j = 0; j < 4; j++) m4_mulv(a, b.c[j], o.c[j]);
    return o;
}
static M4 m4_transpose(const M4& a) {
    M4 o;
    for (int i = 0; i < 4; i++) for (int j = 0; j < 4; j++) o.c[i][j] = a.c[j][i];
    return o;
}
static inline V3 m4_point(const M4& m, V3 p) {          // Matrix4::transform_point
    double v[4] = {p.x, p.y, p.z, 1.0}, o[4];
    m4_mulv(m, v, o);
    double s = 1.0 / o[3];
    return v3(o[0] * s, o[1] * s, o[2] * s);
}
static inline V3 m4_vector(const M4& m, V3 p) {         // Matrix4::transform_vector
    double v[4] = {p.x, p.y, p.z, 0.0}, o[4];
    m4_mulv(m, v, o);
    return v3(o[0], o[1], o[2]);
}

// space/transform.rs:48-190
struct Transform {
    M4 m, minv;
    bool is_identity_bits;   // oracle-side convenience only (never changes results)
    static Transform identity() { return Transform{m4_identity(), m4_identity(), true}; }
    // transform.rs:191-197 concat_self: m = other.m * m ; minv = minv * other.minv
    void concat_self(const Transform& o) {
        M4 nm = m4_mul(o.m, m);
        M4 nminv = m4_mul(minv, o.minv);
        m = nm; minv = nminv; is_identity_bits = false;
    }
};
static Transform t_translate(V3 d) {
    Transform t = Transform::identity();
    t.m.c[3][0] = d.x; t.m.c[3][1] = d.y; t.m.c[3][2] = d.z;
    t.minv.c[3][0] = -d.x; t.minv.c[3][1] = -d.y; t.minv.c[3][2] = -d.z;
    t.is_identity_bits = false;
    return t;
}
static Transform t_scale(double x, double y, double z) {
    Transform t = Transform::identity();
    t.m.c[0][0] = x; t.m.c[1][1] = y; t.m.c[2][2] = z;
    t.minv.c[0][0] = 1.0 / x; t.minv.c[1][1] = 1.0 / y; t.minv.c[2][2] = 1.0 / z;
    t.is_identity_bits = false;
    return t;
}
// cgmath Deg -> Rad: deg * (PI / 180) [assumption: Rad::from(Deg) = deg * PI / 180]
static inline double deg2rad(double d) { return d * PI / 180.0; }
static Transform t_rotate_axis(int axis, double deg) {
    double th = deg2rad(deg), s = std::sin(th), c = std::cos(th);
    M4 m = m4_identity();
    if (axis == 0) { m.c[1][1] = c; m.c[1][2] = s; m.c[2][1] = -s; m.c[2][2] = c; }
    else if (axis == 1) { m.c[0][0] = c; m.c[0][2] = -s; m.c[2][0] = s; m.c[2][2] = c; }
    else { m.c[0][0] = c; m.c[0][1] = s; m.c[1][0] = -s; m.c[1][1] = c; }
    return Transform{m, m4_transpose(m), false};
}
static Transform t_rotate(double deg, V3 a) {   // Matrix4::from_axis_angle (axis not normalised, node.rs:111)
    double th = deg2rad(deg), s = std::sin(th), c = std::cos(th), _1c = 1.0 - c;
    M4 m = m4_identity();
    m.c[0][0] = _1c * a.x * a.x + c;       m.c[0][1] = _1c * a.x * a.y + s * a.z; m.c[0][2] = _1c * a.x * a.z - s * a.y;
    m.c[1][0] = _1c * a.x * a.y - s * a.z; m.c[1][1] = _1c * a.y * a.y + c;       m.c[1][2] = _1c * a.y * a.z + s * a.x;
    m.c[2][0] = _1c * a.x * a.z + s * a.y; m.c[2][1] = _1c * a.y * a.z - s * a.x; m.c[2][2] = _1c * a.z * a.z + c;
    return Transform{m, m4_transpose(m), false};
}

// ---------------------------------------------------------------- ray, bounds
// space/ray.rs:28-33
struct Ray { V3 o, d, dinv; };
static inline Ray ray_new(V3 o, V3 d) { return Ray{o, d, v3(1.0 / d.x, 1.0 / d.y, 1.0 / d.z)}; }

// space/bounds.rs
struct Bounds { V3 mn, mx; };
static inline Bounds b_new(V3 a, V3 b) {              // bounds.rs:37-42
    return Bounds{v3(bmin(a.x, b.x), bmin(a.y, b.y), bmin(a.z, b.z)),
                  v3(bmax(a.x, b.x), bmax(a.y, b.y), bmax(a.z, b.z))};
}
static inline Bounds b_none() { return Bounds{v3(F64_MAX, F64_MAX, F64_MAX), v3(-F64_MAX, -F64_MAX, -F64_MAX)}; }  // :152-157
static inline Bounds b_union(const Bounds& a, const Bounds& b) {   // :55-60
    return Bounds{v3(bmin(a.mn.x, b.mn.x), bmin(a.mn.y, b.mn.y), bmin(a.mn.z, b.mn.z)),
                  v3(bmax(a.mx.x, b.mx.x), bmax(a.mx.y, b.mx.y), bmax(a.mx.z, b.mx.z))};
}
static inline Bounds b_point_union(const Bounds& a, V3 p) {        // :64-69
    return Bounds{v3(bmin(a.mn.x, p.x), bmin(a.mn.y, p.y), bmin(a.mn.z, p.z)),
                  v3(bmax(a.mx.x, p.x), bmax(a.mx.y, p.y), bmax(a.mx.z, p.z))};
}
static inline double b_surface_area(const Bounds& b) {            // :110-114
    V3 d = b.mx - b.mn;
    double half = d.x * d.y + d.x * d.z + d.y * d.z;
    return half + half;
}
static inline int b_maximum_extent(const Bounds& b) {             // :125-130 (sic: d.z > d.z)
    V3 d = b.mx - b.mn;
    if (d.x > d.y && d.z > d.z) return 0;
    else if (d.y > d.z) return 1;
    else return 2;
}
static inline V3 b_offset(const Bounds& b, V3 p) {                // :133-139
    V3 o = p - b.mn;
    if (b.mx.x > b.mn.x) o.x /= b.mx.x - b.mn.x;
    if (b.mx.y > b.mn.y) o.y /= b.mx.y - b.mn.y;
    if (b.mx.z > b.mn.z) o.z /= b.mx.z - b.mn.z;
    return o;
}
// transform.rs:219-240
static Bounds transform_bounds(const Transform& t, const Bounds& b) {
    const M4& m = t.m;
    double xa[3], xb[3], ya[3], yb[3], za[3], zb[3];
    for (int r = 0; r < 3; r++) {
        xa[r] = m.c[0][r] * b.mn.x; xb[r] = m.c[0][r] * b.mx.x;
        ya[r] = m.c[1][r] * b.mn.y; yb[r] = m.c[1][r] * b.mx.y;
        za[r] = m.c[2][r] * b.mn.z; zb[r] = m.c[2][r] * b.mx.z;
    }
    double mn[3], mx[3];
    for (int r = 0; r < 3; r++) {
        mn[r] = bmin(xa[r], xb[r]) + bmin(ya[r], yb[r]) + bmin(za[r], zb[r]);
        mx[r] = bmax(xa[r], xb[r]) + bmax(ya[r], yb[r]) + bmax(za[r], zb[r]);
    }
    V3 pmin = v3(mn[0] + m.c[3][0], mn[1] + m.c[3][1], mn[2] + m.c[3][2]);
    V3 pmax = v3(mx[0] + m.c[3][0], mx[1] + m.c[3][1], mx[2] + m.c[3][2]);
    return b_new(pmin, pmax);
}

// ---------------------------------------------------------------- material
// material/mod.rs:4-46.  One record for the five variants:
//   matte   kd, roughness = sigma (degrees, clamped to [0, 90] by matte.rs:15)
//   plastic kd, ks, roughness
//   metal   kd = eta, ks = k, roughness = u_roughness, roughness2 = v_roughness (metal.rs:13-15)
//   glass   kd = kr, ks = kt, roughness = eta (mod.rs:36-41: the two glass roughnesses are always 0)
//   mirror  kd = kr
enum MatKind { MAT_MATTE = 0, MAT_PLASTIC = 1, MAT_METAL = 2, MAT_GLASS = 3, MAT_MIRROR = 4 };
struct Material { int kind; V3 kd, ks; double roughness; double roughness2 = 0.0; };
static Material mat_default() { return Material{MAT_MATTE, v3(0.5, 0.5, 0.5), v3(0, 0, 0), 0.0}; }   // mod.rs:15-17

// ---------------------------------------------------------------- intersection record
// interaction/surface.rs:33-119
struct RayIsect {
    double t;
    V3 g_dpdu, g_dpdv;     // geometry shading
    V3 s_dpdu, s_dpdv;     // surface shading
    Material material;
    bool has_n; V3 n;
    // oracle-side bookkeeping (AOV only): canonical id of the primitive that wrote the record
    uint32_t prim_id;
};
static inline RayIsect isect_new(double t, V3 dpdu, V3 dpdv) {    // surface.rs:57-62
    RayIsect r; r.t = t; r.g_dpdu = dpdu; r.g_dpdv = dpdv; r.s_dpdu = dpdu; r.s_dpdv = dpdv;
    r.material = mat_default(); r.has_n = false; r.n = v3(0, 0, 0); r.prim_id = 0xFFFFFFFFu;
    return r;
}
static inline RayIsect isect_default() { return isect_new(INF, v3(0, 0, 0), v3(0, 0, 0)); }   // :65-72
static inline V3 isect_ng(const RayIsect& i) { return normalize(cross(i.g_dpdu, i.g_dpdv)); }  // :107-109
static inline V3 isect_ns(const RayIsect& i) {                                                   // :112-118
    if (i.has_n) return normalize(i.n);
    return normalize(cross(i.s_dpdu, i.s_dpdv));
}
static inline void isect_swap_backface(RayIsect& i) {             // :88-99
    std::swap(i.g_dpdu, i.g_dpdv);
    std::swap(i.s_dpdu, i.s_dpdv);
    if (i.has_n) i.n = -i.n;
}
static inline V3 face_forward(V3 n, V3 v) { return dot(n, v) < 0.0 ? -n : n; }   // space/normal.rs:37-40

// transform.rs:243-264
static RayIsect transform_isect(const Transform& t, const RayIsect& i) {
    RayIsect o = isect_new(i.t, m4_vector(t.m, i.g_dpdu), m4_vector(t.m, i.g_dpdv));
    o.material = i.material; o.prim_id = i.prim_id;
    if (!eq(i.g_dpdu, i.s_dpdu) || !eq(i.g_dpdv, i.s_dpdv)) {
        o.s_dpdu = m4_vector(t.m, i.s_dpdu); o.s_dpdv = m4_vector(t.m, i.s_dpdv);
    }
    if (i.has_n) {   // transform_normal :203-210  (minv[col][row] indexing as written in the reference)
        const M4& mi = t.minv; V3 n = i.n;
        o.has_n = true;
        o.n = v3(mi.c[0][0] * n.x + mi.c[0][1] * n.y + mi.c[0][2] * n.z,
                 mi.c[1][0] * n.x + mi.c[1][1] * n.y + mi.c[1][2] * n.z,
                 mi.c[2][0] * n.x + mi.c[2][1] * n.y + mi.c[2][2] * n.z);
    }
    return o;
}
// transform.rs:286-305 (note: the material is NOT carried into the local record)
static RayIsect inverse_transform_isect(const Transform& t, const RayIsect& i) {
    RayIsect o = isect_new(i.t, m4_vector(t.minv, i.g_dpdu), m4_vector(t.minv, i.g_dpdv));
    o.prim_id = i.prim_id;
    if (!eq(i.g_dpdu, i.s_dpdu) || !eq(i.g_dpdv, i.s_dpdv)) {
        o.s_dpdu = m4_vector(t.minv, i.s_dpdu); o.s_dpdv = m4_vector(t.minv, i.s_dpdv);
    }
    if (i.has_n) {   // inverse_transform_normal :267-274
        const M4& m = t.m; V3 n = i.n;
        o.has_n = true;
        o.n = v3(m.c[0][0] * n.x + m.c[0][1] * n.y + m.c[0][2] * n.z,
                 m.c[1][0] * n.x + m.c[1][1] * n.y + m.c[1][2] * n.z,
                 m.c[2][0] * n.x + m.c[2][1] * n.y + m.c[2][2] * n.z);
    }
    return o;
}

// ---------------------------------------------------------------- counters
struct Counters {
    uint64_t node_tests = 0, sphere_tests = 0, cuboid_tests = 0, tri_tests = 0;
    uint64_t primary = 0, primary_hits = 0, shadow = 0, shadow_occluded = 0, exact_ties = 0, secondary = 0;
    void add(const Counters& o) {
        node_tests += o.node_tests; sphere_tests += o.sphere_tests; cuboid_tests += o.cuboid_tests;
        tri_tests += o.tri_tests; primary += o.primary; primary_hits += o.primary_hits;
        shadow += o.shadow; shadow_occluded += o.shadow_occluded; exact_ties += o.exact_ties;
    }
};
static thread_local Counters* g_cnt = nullptr;

// ---------------------------------------------------------------- primitives
// primitive/mod.rs:8-38
struct Primitive {
    virtual ~Primitive() {}
    virtual Bounds bound() const = 0;
    // Returns the innermost primitive hit (nullptr = None).
    virtual const Primitive* intersect(const Ray& ray, RayIsect& isect) const = 0;
    virtual bool material(Material& out) const { (void)out; return false; }
};

// core/math.rs:7-30
static inline int quad_roots(double a, double b, double c, double roots[2]) {
    const double NaN = std::numeric_limits<double>::quiet_NaN();
    if (a == 0.0) {
        if (b == 0.0) { roots[0] = NaN; roots[1] = NaN; return 0; }
        roots[0] = -c / b; roots[1] = NaN; return 1;
    }
    double d = b * b - 4.0 * a * c;
    if (d < 0.0) { roots[0] = NaN; roots[1] = NaN; return 0; }
    double sg = std::signbit(b) ? -1.0 : 1.0;          // f64::signum (NaN aside)
    if (b != b) sg = NaN;
    double q = -(b + sg * std::sqrt(d)) / 2.0;
    double q_over_a = q / a;
    roots[0] = q_over_a;
    roots[1] = (q == 0.0) ? q_over_a : c / q;
    return 2;
}

// shape/sphere.rs
struct Sphere : Primitive {
    V3 origin; double radius; Material mat; uint32_t id;
    // sphere.rs:30-69
    double intersect_t(const Ray& ray, bool& inside) const {
        V3 d = ray.d;
        double rad = radius;
        V3 l = ray.o - origin;
        double a = dot(d, d);
        double b = 2.0 * dot(d, l);
        double c = dot(l, l) - rad * rad;
        double roots[2];
        int n = quad_roots(a, b, c, roots);
        inside = false;
        if (n == 2) {
            double t0 = rmin(roots[0], roots[1]), t1 = rmax(roots[0], roots[1]);
            if (t0 < 0.0) { inside = true; return t1; }
            return t0;
        } else if (n == 1) {
            return roots[0];
        }
        return -INF;
    }
    Bounds bound() const override {                                // :73-77
        return b_new(origin - v3(radius, radius, radius), origin + v3(radius, radius, radius));
    }
    const Primitive* intersect(const Ray& ray, RayIsect& isect) const override {   // :79-123
        if (g_cnt) g_cnt->sphere_tests++;
        bool inside;
        double t = intersect_t(ray, inside);
        if (t < 0.0) return nullptr;
        if (t >= isect.t) { if (g_cnt && t == isect.t) g_cnt->exact_ties++; return nullptr; }
        V3 p = ray.o + ray.d * t - origin;
        if (p.x == 0.0 && p.y == 0.0) p.x = 1e-5 * radius;
        double phi = std::atan2(p.y, p.x);
        if (phi < 0.0) phi += 2.0 * PI;
        double theta = std::acos(rmin(rmax(p.z / radius, -1.0), 1.0));
        V3 dpdu = v3(-2.0 * PI * p.y, 2.0 * PI * p.x, 0.0);
        V3 dpdv = PI * v3(p.z * std::cos(phi), p.z * std::sin(phi), -radius * std::sin(theta));
        if (!inside) std::swap(dpdu, dpdv);
        isect = isect_new(t, dpdu, dpdv);
        isect.prim_id = id;
        return this;
    }
    bool material(Material& out) const override { out = mat; return true; }
};

// shape/cuboid.rs:126-130
static const V3 CUBE_DIFF[3][2] = {
    {{0.0, 1.0, 0.0}, {0.0, 0.0, 1.0}},
    {{0.0, 0.0, 1.0}, {1.0, 0.0, 0.0}},
    {{1.0, 0.0, 0.0}, {0.0, 1.0, 0.0}},
};
// cuboid.rs:104-121 — the BVH node test.  Never looks at isect.t.
static inline bool bounds_intersects(const Bounds& b, const Ray& ray) {
    if (g_cnt) g_cnt->node_tests++;
    double tnear = -INF, tfar = INF;
    for (int i = 0; i < 3; i++) {
        double t1 = (b.mn[i] - ray.o[i]) * ray.dinv[i];
        double t2 = (b.mx[i] - ray.o[i]) * ray.dinv[i];
        double tmin = rmin(t1, t2), tmax = rmax(t1, t2);
        tnear = rmax(tnear, tmin);
        tfar = rmin(tfar, tmax);
    }
    return tnear <= tfar && tfar > 0.0;
}
// cuboid.rs:55-102
static inline bool bounds_intersect(const Bounds& b, const Ray& ray, RayIsect& isect) {
    double tnear = -INF, tfar = INF;
    V3 near0 = CUBE_DIFF[0][0], near1 = CUBE_DIFF[0][1];
    V3 far0 = CUBE_DIFF[0][0], far1 = CUBE_DIFF[0][1];
    for (int i = 0; i < 3; i++) {
        double t1 = (b.mn[i] - ray.o[i]) * ray.dinv[i];
        double t2 = (b.mx[i] - ray.o[i]) * ray.dinv[i];
        double tmin, tmax; V3 dp0, dp1;
        if (t1 < t2) { tmin = t1; tmax = t2; dp0 = CUBE_DIFF[i][1]; dp1 = CUBE_DIFF[i][0]; }
        else { tmin = t2; tmax = t1; dp0 = CUBE_DIFF[i][0]; dp1 = CUBE_DIFF[i][1]; }
        if (tmin > tnear) { near0 = dp0; near1 = dp1; }
        if (tmax < tfar) { far0 = dp1; far1 = dp0; }
        tnear = rmax(tnear, tmin);
        tfar = rmin(tfar, tmax);
    }
    if (tnear > tfar || tfar <= 0.0) return false;
    double t; V3 d0, d1;
    if (tnear <= 0.0) { t = tfar; d0 = far0; d1 = far1; } else { t = tnear; d0 = near0; d1 = near1; }
    if (t >= isect.t) { if (g_cnt && t == isect.t) g_cnt->exact_ties++; return false; }
    isect = isect_new(t, d0, d1);
    isect.has_n = true;
    isect.n = face_forward(cross(d0, d1), -ray.d);
    return true;
}
struct Cuboid : Primitive {
    Bounds bounds; Material mat; uint32_t id;
    Bounds bound() const override { return bounds; }
    const Primitive* intersect(const Ray& ray, RayIsect& isect) const override {
        if (g_cnt) g_cnt->cuboid_tests++;
        if (bounds_intersect(bounds, ray, isect)) { isect.prim_id = id; return this; }
        return nullptr;
    }
    bool material(Material& out) const override { out = mat; return true; }
};

// In-memory result of the `obj` crate for one file: f32 positions / normals and
// polygons (first three IndexTuples only are ever used, triangle.rs:40-55).
struct Mesh {
    std::vector<float> pos;      // 3 * nv
    std::vector<float> nrm;      // 3 * nn (may be empty => has_n() false, triangle.rs:118-120)
    std::vector<uint32_t> vi;    // 3 * ntri position indices
    std::vector<uint32_t> ni;    // 3 * ntri normal indices (iff nrm non-empty)
    size_t ntri() const { return vi.size() / 3; }
};
// space/mod.rs:33-36
static inline int max_dimension(V3 v) {
    if (v.x > v.y) { return v.x > v.z ? 0 : 2; }
    else { return v.y > v.z ? 1 : 2; }
}
// space/mod.rs:39-47
static inline void coordinate_system(V3 v1, V3& v2, V3& v3o) {
    if (std::fabs(v1.x) > std::fabs(v1.y)) v2 = v3(-v1.z, 0.0, v1.x) / std::sqrt(v1.x * v1.x + v1.z * v1.z);
    else v2 = v3(0.0, v1.z, -v1.y) / std::sqrt(v1.y * v1.y + v1.z * v1.z);
    v3o = cross(v1, v2);
}
// shape/triangle.rs
struct Triangle : Primitive {
    const Mesh* mesh; uint32_t tri; uint32_t id;
    V3 p(int k) const { const float* v = &mesh->pos[3 * (size_t)mesh->vi[3 * (size_t)tri + k]]; return v3((double)v[0], (double)v[1], (double)v[2]); }
    V3 n(int k) const { const float* v = &mesh->nrm[3 * (size_t)mesh->ni[3 * (size_t)tri + k]]; return v3((double)v[0], (double)v[1], (double)v[2]); }
    bool has_n() const { return !mesh->nrm.empty(); }
    Bounds bound() const override { return b_point_union(b_new(p(0), p(1)), p(2)); }   // :157-159
    const Primitive* intersect(const Ray& ray, RayIsect& isect) const override {       // :161-307
        if (g_cnt) g_cnt->tri_tests++;
        V3 p0 = p(0), p1 = p(1), p2 = p(2);
        V3 p0t = p0 - ray.o, p1t = p1 - ray.o, p2t = p2 - ray.o;
        int kz = max_dimension(v3(std::fabs(ray.d.x), std::fabs(ray.d.y), std::fabs(ray.d.z)));
        int kx = (kz + 1) % 3;
        int ky = (kx + 1) % 3;
        V3 d = v3(ray.d[kx], ray.d[ky], ray.d[kz]);
        p0t = v3(p0t[kx], p0t[ky], p0t[kz]);
        p1t = v3(p1t[kx], p1t[ky], p1t[kz]);
        p2t = v3(p2t[kx], p2t[ky], p2t[kz]);
        double sx = -d.x / d.z, sy = -d.y / d.z, sz = 1.0 / d.z;
        p0t.x += sx * p0t.z; p0t.y += sy * p0t.z;
        p1t.x += sx * p1t.z; p1t.y += sy * p1t.z;
        p2t.x += sx * p2t.z; p2t.y += sy * p2t.z;
        double e0 = p1t.x * p2t.y - p1t.y * p2t.x;
        double e1 = p2t.x * p0t.y - p2t.y * p0t.x;
        double e2 = p0t.x * p1t.y - p0t.y * p1t.x;
        if ((e0 < 0.0 || e1 < 0.0 || e2 < 0.0) && (e0 > 0.0 || e1 > 0.0 || e2 > 0.0)) return nullptr;
        double det = e0 + e1 + e2;
        if (det == 0.0) return nullptr;
        p0t.z *= sz; p1t.z *= sz; p2t.z *= sz;
        double tscaled = e0 * p0t.z + e1 * p1t.z + e2 * p2t.z;
        if ((det < 0.0 && tscaled >= 0.0) || (det > 0.0 && tscaled <= 0.0)) return nullptr;
        double invdet = 1.0 / det;
        double b0 = e0 * invdet, b1 = e1 * invdet, b2 = e2 * invdet;
        double t = tscaled * invdet;
        if (t >= isect.t) { if (g_cnt && t == isect.t) g_cnt->exact_ties++; return nullptr; }
        // Default uvs (0,0) (1,0) (1,1): no texture coordinates on this path (triangle.rs:80-90).
        double uv[3][2] = {{0.0, 0.0}, {1.0, 0.0}, {1.0, 1.0}};
        double duv02x = uv[0][0] - uv[2][0], duv02y = uv[0][1] - uv[2][1];
        double duv12x = uv[1][0] - uv[2][0], duv12y = uv[1][1] - uv[2][1];
        V3 dp02 = p0 - p2, dp12 = p1 - p2;
        double determinant = (duv02x * duv12y) - (duv02y * duv12x);
        V3 dpdu, dpdv;
        if (determinant == 0.0) {
            coordinate_system(cross(p2 - p1, p1 - p0), dpdu, dpdv);
        } else {
            double inv = 1.0 / determinant;
            dpdu = (duv12y * dp02 - duv02y * dp12) * inv;
            dpdv = (-duv12x * dp02 - duv02x * dp12) * inv;
        }
        isect = isect_new(t, dpdu, dpdv);
        isect.prim_id = id;
        if (has_n()) {                                                                  // :284-299
            V3 ns = b0 * n(0) + b1 * n(1) + b2 * n(2);
            V3 ss = isect.g_dpdu;
            V3 ts = cross(ns, ss);
            if (dot(ts, ts) > 0.0) { ss = cross(ts, ns); }
            else { coordinate_system(ns, ss, ts); }
            isect.has_n = true; isect.n = ns;
            isect.s_dpdu = ss; isect.s_dpdv = ts;
        } else {                                                                        // :300-304
            isect.has_n = true;
            isect.n = face_forward(cross(dp02, dp12), -ray.d);
        }
        return this;
    }
};

// ---------------------------------------------------------------- BVH (accelerators/bvh.rs)
struct LinearNode {           // bvh.rs:119-131
    Bounds bounds;
    bool leaf;
    uint32_t a;               // leaf: prim_offset        interior: second child index
    uint32_t b;               // leaf: nprims (u16)       interior: axis (u8)
};
struct MortonPrim { size_t index; uint32_t code; };
struct BuildNode {            // bvh.rs:95-110
    bool leaf = true; size_t first = 0, n = 0; int axis = 0;
    BuildNode* c0 = nullptr; BuildNode* c1 = nullptr; Bounds bounds = b_none();
};
struct PrimInfo { size_t number; Bounds bounds; V3 centroid; };

static inline uint32_t left_shift_3(uint32_t x) {     // bvh.rs:590-598
    if (x == (1u << 10)) x -= 1;
    x = (x | (x << 16)) & 0b00000011000000000000000011111111u;
    x = (x | (x << 8)) & 0b00000011000000001111000000001111u;
    x = (x | (x << 4)) & 0b00000011000011000011000011000011u;
    x = (x | (x << 2)) & 0b00001001001001001001001001001001u;
    return x;
}
static inline uint32_t encode_morton_3(V3 v) {         // bvh.rs:575-579 (sic: z, y, z)
    return (left_shift_3(as_u32(v.z)) << 2) | (left_shift_3(as_u32(v.y)) << 1) | left_shift_3(as_u32(v.z));
}
static void radix_sort(std::vector<MortonPrim>& v) {   // bvh.rs:600-635
    std::vector<MortonPrim> temp(v.size(), MortonPrim{0, 0});
    const uint32_t bits_per_pass = 6, nbits = 30, npasses = nbits / bits_per_pass, nbuckets = 1u << bits_per_pass;
    const uint32_t mask = (1u << bits_per_pass) - 1;
    for (uint32_t pass = 0; pass < npasses; pass++) {
        uint32_t lowbit = pass * bits_per_pass;
        std::vector<MortonPrim>& in = (pass & 1) == 0 ? v : temp;
        std::vector<MortonPrim>& out = (pass & 1) == 0 ? temp : v;
        size_t count[64] = {0};
        for (const MortonPrim& mp : in) count[(mp.code >> lowbit) & mask]++;
        size_t out_index[64]; out_index[0] = 0;
        for (uint32_t i = 1; i < nbuckets; i++) out_index[i] = out_index[i - 1] + count[i - 1];
        for (const MortonPrim& mp : in) out[out_index[(mp.code >> lowbit) & mask]++] = mp;
    }
    if (npasses & 1) std::swap(v, temp);
}

struct Scene;
struct BVH : Primitive {
    const Scene* scene = nullptr;
    std::vector<std::unique_ptr<Primitive>> primitives;
    std::vector<LinearNode> nodes;
    Transform transform = Transform::identity();
    std::vector<size_t> order;
    bool has_material = false; Material mat;
    uint8_t max_prims_per_node = 0;
    bool swap_backface = false;
    std::vector<std::unique_ptr<BuildNode[]>> arena;     // typed_arena stand-in
    bool build_failed = false;

    BuildNode* alloc(size_t n) { arena.emplace_back(new BuildNode[n]); return arena.back().get(); }

    // bvh.rs:164-202
    void init(size_t per_node) {
        size_t nprims = primitives.size();
        std::vector<PrimInfo> info(nprims);
        for (size_t i = 0; i < nprims; i++) {           // :525-532
            Bounds b = primitives[i]->bound();
            info[i] = PrimInfo{i, b, 0.5 * b.mn + 0.5 * b.mx};
        }
        order.assign(nprims, SIZE_MAX);
        max_prims_per_node = (uint8_t)std::min<size_t>(per_node, 255);
        size_t total_nodes = 0;
        BuildNode* root = build(info, total_nodes);
        if (!root) { build_failed = true; return; }
        nodes.assign(total_nodes, LinearNode{b_none(), true, 0, 0});
        size_t off = 0;
        flatten(root, off);
        arena.clear();
    }
    // bvh.rs:205-273
    BuildNode* build(const std::vector<PrimInfo>& info, size_t& total_nodes) {
        if (info.empty()) return nullptr;                // Q9: the reference recurses forever
        Bounds bounds = b_none();
        for (const PrimInfo& pi : info) bounds = b_union(bounds, pi.bounds);
        std::vector<MortonPrim> mp(info.size());
        for (size_t i = 0; i < info.size(); i++) {
            V3 off = b_offset(bounds, info[i].centroid);
            mp[i] = MortonPrim{info[i].number, encode_morton_3(off * 1024.0)};
        }
        radix_sort(mp);
        std::vector<BuildNode*> treelets;
        size_t start = 0, ordered_off = 0, total = 0;
        const uint32_t mask = 0b00111111111111000000000000000000u;
        for (size_t end = 1; end <= mp.size(); end++) {
            if (end == mp.size() || ((mp[start].code & mask) != (mp[end].code & mask))) {
                size_t created = 0, nprims = end - start;
                BuildNode* nodes_buf = alloc(2 * nprims);
                BuildNode* next = nodes_buf;
                BuildNode* node = emit_lbvh(next, &mp[start], nprims, info, created, ordered_off, 29 - 12);
                total += created;
                treelets.push_back(node);
                start = end;
            }
        }
        total_nodes += total;
        int depth_guard = 0;
        return build_upper_sah(treelets.data(), treelets.size(), total_nodes, depth_guard);
    }
    // bvh.rs:278-347
    BuildNode* emit_lbvh(BuildNode*& next, const MortonPrim* mp, size_t nprims, const std::vector<PrimInfo>& info,
                         size_t& total_nodes, size_t& ordered_off, int bit_index) {
        if (bit_index == -1 || nprims < (size_t)max_prims_per_node) {
            size_t first = ordered_off;
            BuildNode* node = next++;
            ordered_off += nprims;
            total_nodes += 1;
            Bounds b = b_none();
            for (size_t i = 0; i < nprims; i++) {
                size_t pi = mp[i].index;
                order[first + i] = pi;
                b = b_union(b, info[pi].bounds);
            }
            node->leaf = true; node->first = first; node->n = nprims; node->bounds = b;
            return node;
        }
        uint32_t mask = 1u << bit_index;
        if ((mp[0].code & mask) == (mp[nprims - 1].code & mask))
            return emit_lbvh(next, mp, nprims, info, total_nodes, ordered_off, bit_index - 1);
        size_t s = 0, e = nprims - 1;
        while (s + 1 != e) {
            size_t mid = (s + e) / 2;
            if ((mp[s].code & mask) == (mp[mid].code & mask)) s = mid; else e = mid;
        }
        size_t split = e;
        BuildNode* node = next++;
        total_nodes += 1;
        BuildNode* l0 = emit_lbvh(next, mp, split, info, total_nodes, ordered_off, bit_index - 1);
        BuildNode* l1 = emit_lbvh(next, mp + split, nprims - split, info, total_nodes, ordered_off, bit_index - 1);
        node->leaf = false; node->axis = bit_index % 3; node->c0 = l0; node->c1 = l1;
        node->bounds = b_union(l0->bounds, l1->bounds);    // :557-560
        return node;
    }
    // bvh.rs:350-427
    BuildNode* build_upper_sah(BuildNode** roots, size_t ncount, size_t& total_nodes, int& depth) {
        if (ncount == 1) return roots[0];
        if (ncount == 0 || depth > 4096) return nullptr;   // Q9/Q10: the reference would not terminate
        BuildNode* node = alloc(1);
        total_nodes += 1;
        Bounds bounds = b_none(), cb = b_none();
        for (size_t i = 0; i < ncount; i++) bounds = b_union(bounds, roots[i]->bounds);
        for (size_t i = 0; i < ncount; i++) {
            V3 c = 0.5 * (roots[i]->bounds.mn + roots[i]->bounds.mx);
            cb = b_point_union(cb, c);
        }
        int dim = b_maximum_extent(cb);
        const int NB = 12;
        size_t bcount[NB]; Bounds bb[NB];
        for (int i = 0; i < NB; i++) { bcount[i] = 0; bb[i] = b_none(); }
        auto bucket_of = [&](const BuildNode* r, bool half_first) -> size_t {
            // :383 uses (min+max)*0.5, :415 uses 0.5*(min+max): identical products.
            double centroid = half_first ? 0.5 * (r->bounds.mn[dim] + r->bounds.mx[dim])
                                         : (r->bounds.mn[dim] + r->bounds.mx[dim]) * 0.5;
            double b0 = (centroid - cb.mn[dim]) / (cb.mx[dim] - cb.mn[dim]);
            size_t b = (size_t)as_u32((double)NB * b0);
            if (b == (size_t)NB) b = NB - 1;
            return b;
        };
        for (size_t i = 0; i < ncount; i++) {
            size_t b = bucket_of(roots[i], false);
            if (b >= (size_t)NB) return nullptr;           // Rust would panic on the index
            bcount[b] += 1;
            bb[b] = b_union(bb[b], roots[i]->bounds);
        }
        double cost[NB];
        for (int i = 0; i < NB; i++) {
            Bounds b0 = b_none(), b1 = b_none(); size_t c0 = 0, c1 = 0;
            for (int j = 0; j <= i; j++) { b0 = b_union(b0, bb[j]); c0 += bcount[j]; }
            for (int j = i + 1; j < NB; j++) { b1 = b_union(b1, bb[j]); c1 += bcount[j]; }
            cost[i] = 0.125 + ((double)c0 * b_surface_area(b0) + (double)c1 * b_surface_area(b1)) / b_surface_area(bounds);
        }
        int min_bucket = 0;
        for (int i = 0; i < NB; i++) if (cost[i] < cost[min_bucket]) min_bucket = i;
        // `partition` crate: predicate-true elements first.  Order inside each side
        // never influences the tree (only min/max/count folds consume it).
        BuildNode** mid = std::partition(roots, roots + ncount, [&](BuildNode* r) {
            return bucket_of(r, true) <= (size_t)min_bucket;
        });
        size_t nlo = (size_t)(mid - roots);
        if (nlo == 0 || nlo == ncount) return nullptr;     // Q10: the reference recurses forever
        depth++;
        BuildNode* lo = build_upper_sah(roots, nlo, total_nodes, depth);
        BuildNode* hi = lo ? build_upper_sah(mid, ncount - nlo, total_nodes, depth) : nullptr;
        depth--;
        if (!lo || !hi) return nullptr;
        node->leaf = false; node->axis = dim; node->c0 = lo; node->c1 = hi;
        node->bounds = b_union(lo->bounds, hi->bounds);
        return node;
    }
    // bvh.rs:430-453
    size_t flatten(const BuildNode* node, size_t& offset) {
        size_t my = offset++;
        nodes[my].bounds = node->bounds;
        if (node->leaf) {
            nodes[my].leaf = true; nodes[my].a = (uint32_t)node->first; nodes[my].b = (uint32_t)(uint16_t)node->n;
        } else {
            flatten(node->c0, offset);
            size_t second = flatten(node->c1, offset);
            nodes[my].leaf = false; nodes[my].a = (uint32_t)second; nodes[my].b = (uint32_t)(uint8_t)node->axis;
        }
        return my;
    }

    Bounds bound() const override { return transform_bounds(transform, nodes[0].bounds); }   // :457-459
    // bvh.rs:461-522
    const Primitive* intersect(const Ray& ray_in, RayIsect& isect) const override {
        Ray ray = ray_new(m4_point(transform.minv, ray_in.o), m4_vector(transform.minv, ray_in.d));   // transform.rs:279-283
        bool dir_is_neg[3] = {ray.dinv.x < 0.0, ray.dinv.y < 0.0, ray.dinv.z < 0.0};
        RayIsect isect_inv = inverse_transform_isect(transform, isect);
        const Primitive* hit = nullptr;
        size_t to_visit = 0, cur = 0;
        size_t stack[64];
        for (;;) {
            const LinearNode& node = nodes[cur];
            if (!bounds_intersects(node.bounds, ray)) {
                if (to_visit == 0) break;
                cur = stack[--to_visit];
                continue;
            }
            if (node.leaf) {
                for (uint32_t i = 0; i < node.b; i++) {
                    size_t pi = order[(size_t)node.a + i];
                    const Primitive* p = primitives[pi]->intersect(ray, isect_inv);
                    if (p) hit = p;
                }
                if (to_visit == 0) break;
                cur = stack[--to_visit];
            } else {
                if (to_visit >= 64) { stack_overflow.store(true); break; }   // Q8: Rust panics here
                if (dir_is_neg[node.b]) { stack[to_visit] = cur + 1; cur = node.a; }
                else { stack[to_visit] = node.a; cur += 1; }
                to_visit++;
            }
        }
        if (hit) {
            isect = transform_isect(transform, isect_inv);
            if (has_material) isect.material = mat;
            if (swap_backface) isect_swap_backface(isect);
        }
        return hit;
    }
    mutable std::atomic<bool> stack_overflow{false};
};

// ---------------------------------------------------------------- scene (scene.rs, scene/node.rs)
enum NodeKind { N_SPHERE, N_CUBE, N_CUBOID, N_MESH, N_GROUP };
struct SceneNode {
    NodeKind kind; V3 a, b; double r; Material mat; bool has_mat; int ref;   // ref: mesh index or aggregate index
};
struct Aggregate { std::vector<SceneNode> contents; Transform transform = Transform::identity(); bool swap_backface = false; };

struct Camera {                // camera.rs
    V3 origin{0, 0, 0}, view{0, 0, 1}, up{0, 1, 0}, aux{1, 0, 0};
    bool perspective = true; double param = 45.0;     // fov (deg) or orthographic height
    size_t root = 1; double distance = 1.0;           // Supersampling :177-193
    double image_plane_height = 0.0, pixel_separation = 0.0;
    double plane_height(double focal) const {           // :158-164
        return perspective ? focal * std::tan(param * PI / 360.0) * 2.0 : param;
    }
    void reset(bool persp, double p) {                  // :61-73
        perspective = persp; param = p;
        origin = v3(0, 0, 0); view = v3(0, 0, 1); up = v3(0, 1, 0); aux = v3(1, 0, 0);
        root = 1; distance = 1.0;
        image_plane_height = plane_height(1.0);
        pixel_separation = persp ? 0.0 : 1.0;
    }
    void look_at(V3 o, V3 look, V3 upv) {               // :85-94
        V3 v = look - o;
        V3 ax = cross(v, upv);
        origin = o;
        up = normalize(cross(ax, v));
        aux = normalize(ax);
        view = v;
        image_plane_height = plane_height(magnitude(v));
    }
    void set_supersampling(uint8_t base) { root = (size_t)base + 1; distance = 1.0 / (double)root; }   // :189-193
};
struct Light { V3 position, intensity; double falloff[3]; };
struct Background { V3 inner, outer; double scale; };

struct Scene {
    std::vector<Aggregate> aggs;            // aggs[0] = root; groups are referenced by index
    Camera camera;
    Background background{v3(0, 0, 0), v3(0, 0, 0), 1.0};
    V3 ambient{0, 0, 0};
    uint32_t recursion = 3;
    std::vector<Light> lights;
    std::vector<Mesh> meshes;
    Scene() { aggs.emplace_back(); camera.reset(true, 45.0); }
};

struct Accel {
    const Scene* scene;
    std::unique_ptr<BVH> root;
    uint32_t next_id = 0;
    bool failed = false;
    double build_ms = 0.0;
    // bvh.rs:141-148
    std::unique_ptr<BVH> from_mesh(int mesh, bool has_mat, Material mat) {
        auto bvh = std::make_unique<BVH>();
        bvh->scene = scene;
        const Mesh& m = scene->meshes[mesh];
        for (size_t i = 0; i < m.ntri(); i++) {
            auto t = std::make_unique<Triangle>();
            t->mesh = &m; t->tri = (uint32_t)i; t->id = next_id++;
            bvh->primitives.push_back(std::move(t));
        }
        bvh->has_material = has_mat; bvh->mat = mat;
        bvh->init(m.ntri());
        if (bvh->build_failed) failed = true;
        return bvh;
    }
    // bvh.rs:150-162
    std::unique_ptr<BVH> from_aggregate(int ai) {
        const Aggregate& ag = scene->aggs[ai];
        auto bvh = std::make_unique<BVH>();
        bvh->scene = scene;
        for (const SceneNode& n : ag.contents) {
            switch (n.kind) {
            case N_SPHERE: { auto s = std::make_unique<Sphere>(); s->origin = n.a; s->radius = n.r; s->mat = n.mat; s->id = next_id++; bvh->primitives.push_back(std::move(s)); break; }
            case N_CUBE: { auto c = std::make_unique<Cuboid>(); c->bounds = b_new(n.a, n.a + v3(n.r, n.r, n.r)); c->mat = n.mat; c->id = next_id++; bvh->primitives.push_back(std::move(c)); break; }   // cuboid.rs:24-30
            case N_CUBOID: { auto c = std::make_unique<Cuboid>(); c->bounds = b_new(n.a, n.b); c->mat = n.mat; c->id = next_id++; bvh->primitives.push_back(std::move(c)); break; }              // cuboid.rs:18-22
            case N_MESH: { auto m = from_mesh(n.ref, n.has_mat, n.mat); if (failed) return bvh; bvh->primitives.push_back(std::move(m)); break; }
            case N_GROUP: { auto g = from_aggregate(n.ref); if (failed) return bvh; bvh->primitives.push_back(std::move(g)); break; }
            }
        }
        bvh->transform = ag.transform;
        bvh->swap_backface = ag.swap_backface;
        bvh->init(bvh->primitives.size());
        if (bvh->build_failed) failed = true;
        return bvh;
    }
};

// ---------------------------------------------------------------- shading
// core/bxdf/mod.rs:237-258
static inline double cos2_theta(V3 w) { return w.z * w.z; }
static inline double sin2_theta(V3 w) { return rmax(1.0 - cos2_theta(w), 0.0); }
static inline double sin_theta(V3 w) { return std::sqrt(sin2_theta(w)); }
static inline double tan_theta(V3 w) { return sin_theta(w) / w.z; }
static inline double tan2_theta(V3 w) { return sin2_theta(w) / cos2_theta(w); }
static inline double cos_phi(V3 w) { double s = sin_theta(w); return s == 0.0 ? 1.0 : rmin(rmax(w.x / s, -1.0), 1.0); }
static inline double sin_phi(V3 w) { double s = sin_theta(w); return s == 0.0 ? 0.0 : rmin(rmax(w.y / s, -1.0), 1.0); }
static inline double cos2_phi(V3 w) { return cos_phi(w) * cos_phi(w); }
static inline double sin2_phi(V3 w) { return sin_phi(w) * sin_phi(w); }

// core/bxdf/fresnel.rs:37-64
static double dielectric(double cos_theta_i, double eta_i, double eta_t) {
    cos_theta_i = rmin(rmax(cos_theta_i, -1.0), 1.0);
    bool entering = cos_theta_i > 0.0;
    if (!entering) { std::swap(eta_i, eta_t); cos_theta_i = std::fabs(cos_theta_i); }
    double sin_theta_i = std::sqrt(rmax(1.0 - cos_theta_i * cos_theta_i, 0.0));
    double sin_theta_t = eta_i / eta_t * sin_theta_i;
    if (sin_theta_t >= 1.0) return 1.0;
    double cos_theta_t = std::sqrt(rmax(1.0 - sin_theta_t * sin_theta_t, 0.0));
    double r_parl = ((eta_t * cos_theta_i) - (eta_i * cos_theta_t)) / ((eta_t * cos_theta_i) + (eta_i * cos_theta_t));
    double r_perp = ((eta_i * cos_theta_i) - (eta_t * cos_theta_t)) / ((eta_i * cos_theta_i) + (eta_t * cos_theta_t));
    return (r_parl * r_parl + r_perp * r_perp) * 0.5;
}
// core/bxdf/microfacet.rs:31-66
struct Distribution {
    double ax, ay;
    double d(V3 wh) const {
        double t2 = tan2_theta(wh);
        if (std::isinf(t2)) return 0.0;
        double cos4 = cos2_theta(wh) * cos2_theta(wh);
        double e = (cos2_phi(wh) / (ax * ax) + sin2_phi(wh) / (ay * ay)) * t2;
        return 1.0 / (PI * ax * ay * cos4 * (1.0 + e) * (1.0 + e));
    }
    double lambda(V3 w) const {
        double att = std::fabs(tan_theta(w));
        if (std::isinf(att)) return 0.0;
        double alpha = std::sqrt(cos2_phi(w) * ax * ax + sin2_phi(w) * ay * ay);
        double a2t2 = (alpha * att) * (alpha * att);
        return (std::sqrt(1.0 + a2t2) - 1.0) / 2.0;
    }
    double g(V3 wo, V3 wi) const { return 1.0 / (1.0 + lambda(wo) + lambda(wi)); }
};
// core/bxdf/fresnel.rs:68-90
static V3 conductor(double cos_theta_i, V3 eta_i, V3 eta_t, V3 k) {
    cos_theta_i = rmin(rmax(cos_theta_i, -1.0), 1.0);
    V3 eta = v3(eta_t.x / eta_i.x, eta_t.y / eta_i.y, eta_t.z / eta_i.z);
    V3 etak = v3(k.x / eta_i.x, k.y / eta_i.y, k.z / eta_i.z);
    double cos2 = cos_theta_i * cos_theta_i;
    double sin2 = 1.0 - cos2;
    V3 eta2 = mul_el(eta, eta), etak2 = mul_el(etak, etak);
    auto chan = [&](double e2, double ek2) {
        double t0 = e2 - ek2 - sin2;
        double a2plusb2 = std::sqrt(t0 * t0 + 4.0 * (e2 * ek2));
        double t1 = a2plusb2 + cos2;
        double a = std::sqrt(0.5 * (a2plusb2 + t0));
        double t2 = 2.0 * cos_theta_i * a;
        double rs = (t1 - t2) / (t1 + t2);
        double t3 = cos2 * a2plusb2 + sin2 * sin2;
        double t4 = t2 * sin2;
        double rp = rs * (t3 - t4) / (t3 + t4);
        return 0.5 * (rp + rs);
    };
    return v3(chan(eta2.x, etak2.x), chan(eta2.y, etak2.y), chan(eta2.z, etak2.z));
}
// core/bxdf/fresnel.rs:7-33
enum SubstKind { SUB_DIELECTRIC = 0, SUB_CONDUCTOR = 1, SUB_NOOP = 2 };
struct Substance {
    int kind = SUB_NOOP; double eta_i = 1.0, eta_t = 1.0; V3 c_eta_i, c_eta_t, c_k;
    V3 evaluate(double cos_theta_i) const {
        if (kind == SUB_DIELECTRIC) { double F = dielectric(cos_theta_i, eta_i, eta_t); return v3(F, F, F); }
        if (kind == SUB_CONDUCTOR) return conductor(cos_theta_i, c_eta_i, c_eta_t, c_k);
        return v3(1.0, 1.0, 1.0);
    }
};
// microfacet.rs:101-115
static V3 microfacet_f(V3 r, const Substance& sub, const Distribution& dist, V3 wo, V3 wi) {
    double cos_o = std::fabs(wo.z), cos_i = std::fabs(wi.z);
    V3 wh = wi + wo;
    if (cos_i == 0.0 || cos_o == 0.0) return v3(0, 0, 0);
    if (wh.x == 0.0 && wh.y == 0.0 && wh.z == 0.0) return v3(0, 0, 0);
    wh = normalize(wh);
    V3 spectrum = sub.evaluate(dot(wi, wh));
    return mul_el(r * dist.d(wh) * dist.g(wo, wi), spectrum) / (4.0 * cos_i * cos_o);
}

// interaction/surface.rs:158-183
struct SurfaceInteraction { V3 p, p_err, wo, ng, ns, g_dpdu, g_dpdv, s_dpdu, s_dpdv; };
static SurfaceInteraction surface_from(const Ray& ray, const RayIsect& isect) {
    SurfaceInteraction si;
    si.wo = -normalize(ray.d);
    si.ng = face_forward(isect_ng(isect), si.wo);
    si.ns = isect_ns(isect);
    double err = std::numeric_limits<double>::epsilon() * 65536.0;     // EPSILON * 2^16
    si.p = ray.o + ray.d * isect.t;
    si.p_err = si.ng * err;
    si.g_dpdu = normalize(isect.g_dpdu); si.g_dpdv = normalize(isect.g_dpdv);
    si.s_dpdu = normalize(isect.s_dpdu); si.s_dpdv = normalize(isect.s_dpdv);
    return si;
}
// bxdf/mod.rs:18-31
enum : uint32_t { BX_REFLECTION = 1, BX_TRANSMISSION = 2, BX_DIFFUSE = 4, BX_GLOSSY = 8, BX_SPECULAR = 16 };
enum BxKind { BX_QUICK_DIFFUSE, BX_OREN_NAYAR, BX_MICROFACET_REFLECTION, BX_SPECULAR_REFLECTION, BX_SPECULAR_TRANSMISSION };
struct LightSample { V3 spectrum, wi; double pdf; };
// bxdf/mod.rs:164-174: refract in shading coordinates
static bool refract(V3 wi, V3 n, double eta, V3& out) {
    double cos_i = dot(n, wi);
    double sin2_i = rmax(1.0 - cos_i * cos_i, 0.0);
    double sin2_t = eta * eta * sin2_i;
    if (sin2_t >= 1.0) return false;
    double cos_t = std::sqrt(1.0 - sin2_t);
    out = (eta * -1.0) * wi + (eta * cos_i - cos_t) * n;
    return true;
}
struct BxDF {
    int kind; V3 r; double a = 0, b = 0; Substance sub; Distribution dist{1, 1}; double eta_a = 1, eta_b = 1;
    uint32_t t() const {                                                  // mod.rs:141-152
        switch (kind) {
            case BX_QUICK_DIFFUSE: case BX_OREN_NAYAR: return BX_REFLECTION | BX_DIFFUSE;
            case BX_MICROFACET_REFLECTION: return BX_REFLECTION | BX_GLOSSY;
            case BX_SPECULAR_REFLECTION: return BX_REFLECTION | BX_SPECULAR;
            default: return BX_TRANSMISSION | BX_SPECULAR;
        }
    }
    bool matches(uint32_t flags) const { return (t() & flags) == t(); }  // mod.rs:154-157
    bool has_t(uint32_t flags) const { return (t() & flags) != 0; }      // mod.rs:159-161
    V3 f(V3 wo, V3 wi) const {                                            // mod.rs:165-175
        switch (kind) {
            case BX_QUICK_DIFFUSE: return r * FRAC_1_PI;                  // diffuse.rs:14
            case BX_OREN_NAYAR: {                                         // diffuse.rs:36-56
                double sin_i = sin_theta(wi), sin_o = sin_theta(wo);
                double max_cos = 0.0;
                if (sin_i > 1e-4 && sin_o > 1e-4) {
                    double d_cos = cos_phi(wi) * cos_phi(wo) + sin_phi(wi) * sin_phi(wo);
                    max_cos = rmax(d_cos, 0.0);
                }
                double sin_alpha, tan_beta;
                if (std::fabs(wi.z) > std::fabs(wo.z)) { sin_alpha = sin_o; tan_beta = sin_i / std::fabs(wi.z); }
                else { sin_alpha = sin_i; tan_beta = sin_o / std::fabs(wo.z); }
                return r * FRAC_1_PI * (a + b * max_cos * sin_alpha * tan_beta);
            }
            case BX_MICROFACET_REFLECTION: return microfacet_f(r, sub, dist, wo, wi);
            default: return v3(0, 0, 0);                                  // specular lobes scatter only through sample_f
        }
    }
    // specular.rs:17-25, 44-66 (the only sample_f variants a Whitted path reaches: integrate.rs:85,110)
    LightSample sample_f(V3 wo) const {
        if (kind == BX_SPECULAR_REFLECTION) {
            V3 wi = v3(-wo.x, -wo.y, wo.z);
            V3 spectrum = mul_el(sub.evaluate(wi.z), r) / std::fabs(wi.z);
            return LightSample{spectrum, wi, 1.0};
        }
        bool entering = wo.z > 0.0;
        double eta_i = entering ? eta_a : eta_b, eta_t = entering ? eta_b : eta_a;
        V3 wi;
        if (!refract(wo, v3(0.0, 0.0, 1.0), eta_i / eta_t, wi)) return LightSample{v3(0, 0, 0), v3(0, 0, 0), 0.0};
        V3 spectrum = mul_el(r, v3(1.0, 1.0, 1.0) - sub.evaluate(wi.z)) / std::fabs(wi.z);
        return LightSample{spectrum, wi, 1.0};
    }
};
static BxDF oren_nayar(V3 r, double sigma_deg) {                          // diffuse.rs:28-34
    double sigma = deg2rad(sigma_deg);
    double sigma2 = sigma * sigma;
    BxDF b; b.kind = BX_OREN_NAYAR; b.r = r;
    b.a = 1.0 - (sigma2 / 2.0 * (sigma2 + 0.33));
    b.b = 0.45 * sigma2 / (sigma2 + 0.09);
    return b;
}
// interaction/bsdf.rs:29-46, 73-92, 94-140, 155-175 + material/{matte,plastic,metal,glass,mirror}.rs
struct BSDF {
    V3 ng, ns, ss, ts;
    BxDF bx[2]; int n = 0;
    void add(const BxDF& b) { bx[n++] = b; }
    V3 to_local(V3 v) const { return v3(dot(v, ss), dot(v, ts), dot(v, ns)); }
    V3 to_world(V3 v) const {
        return v3(ss.x * v.x + ts.x * v.y + ns.x * v.z, ss.y * v.x + ts.y * v.y + ns.y * v.z, ss.z * v.x + ts.z * v.y + ns.z * v.z);
    }
    V3 f(V3 wo, V3 wi) const {
        bool reflect = dot(wi, ng) * dot(wo, ng) > 0.0;
        V3 wo_l = to_local(wo), wi_l = to_local(wi);
        if (wo_l.z == 0.0) return v3(0, 0, 0);
        V3 f = v3(0, 0, 0);
        for (int i = 0; i < n; i++)
            if ((reflect && bx[i].has_t(BX_REFLECTION)) || (!reflect && bx[i].has_t(BX_TRANSMISSION))) f = f + bx[i].f(wo_l, wi_l);
        return f;
    }
    // bsdf.rs:94-140 with sample = (0.5, 0.5) and SPECULAR flags: at most one lobe of a material matches either flag set
    // (glass: one reflection + one transmission lobe), so comp = 0 and pdf = f_sample.pdf / 1.
    LightSample sample_f(V3 wo, uint32_t flags) const {
        int matching = 0; const BxDF* pick = nullptr;
        for (int i = 0; i < n; i++) if (bx[i].matches(flags)) { if (!pick) pick = &bx[i]; matching++; }
        if (matching == 0) return LightSample{v3(0, 0, 0), v3(0, 0, 0), 0.0};
        V3 wo_l = to_local(wo);
        if (wo_l.z == 0.0) return LightSample{v3(0, 0, 0), v3(0, 0, 0), 0.0};
        LightSample fs = pick->sample_f(wo_l);
        if (fs.pdf == 0.0) return fs;
        V3 wi = to_world(fs.wi);
        auto clamp01 = [](double v) { return rmin(rmax(v, 0.0), 1.0); };
        V3 spectrum = v3(clamp01(fs.spectrum.x), clamp01(fs.spectrum.y), clamp01(fs.spectrum.z));
        return LightSample{spectrum, wi, fs.pdf / (double)matching};
    }
};
static inline bool is_zero(V3 c) { return c.x == 0.0 && c.y == 0.0 && c.z == 0.0; }
static bool scattering(const Material& m, const SurfaceInteraction& si, BSDF& b) {
    b.ng = si.ng; b.ns = si.ns; b.ss = si.s_dpdu; b.ts = cross(si.ns, b.ss); b.n = 0;
    BxDF x;
    switch (m.kind) {
    case MAT_PLASTIC:                                                      // plastic.rs:20-37
        if (!is_zero(m.kd)) { x.kind = BX_QUICK_DIFFUSE; x.r = m.kd; b.add(x); }
        if (!is_zero(m.ks)) {
            x = BxDF(); x.kind = BX_MICROFACET_REFLECTION; x.r = m.ks; x.sub.kind = SUB_DIELECTRIC; x.sub.eta_i = 1.0; x.sub.eta_t = 1.5;
            x.dist = Distribution{m.roughness, m.roughness}; b.add(x);
        }
        return true;
    case MAT_MATTE:                                                        // matte.rs:18-26
        if (m.roughness == 0.0) { x.kind = BX_QUICK_DIFFUSE; x.r = m.kd; b.add(x); }
        else b.add(oren_nayar(m.kd, m.roughness));
        return true;
    case MAT_METAL:                                                        // metal.rs:17-26
        x.kind = BX_MICROFACET_REFLECTION; x.r = v3(1.0, 1.0, 1.0);
        x.sub.kind = SUB_CONDUCTOR; x.sub.c_eta_i = v3(1.0, 1.0, 1.0); x.sub.c_eta_t = m.kd; x.sub.c_k = m.ks;
        x.dist = Distribution{m.roughness, m.roughness2}; b.add(x);
        return true;
    case MAT_GLASS:                                                        // glass.rs:33-56 (distribution = None)
        if (!is_zero(m.kd)) { x.kind = BX_SPECULAR_REFLECTION; x.r = m.kd; x.sub.kind = SUB_DIELECTRIC; x.sub.eta_i = 1.0; x.sub.eta_t = m.roughness; b.add(x); }
        if (!is_zero(m.ks)) {
            x = BxDF(); x.kind = BX_SPECULAR_TRANSMISSION; x.r = m.ks; x.eta_a = 1.0; x.eta_b = m.roughness;
            x.sub.kind = SUB_DIELECTRIC; x.sub.eta_i = 1.0; x.sub.eta_t = m.roughness; b.add(x);
        }
        return true;
    case MAT_MIRROR:                                                       // mirror.rs:14-16
        x.kind = BX_SPECULAR_REFLECTION; x.r = m.kd; x.sub.kind = SUB_NOOP; b.add(x);
        return true;
    }
    return false;
}
static inline double lerp(double t, double a, double b) { return a * (1.0 - t) + b * t; }    // space/mod.rs:28-30
// material/background.rs:25-34  (powf(2.) folded to x*x, as LLVM does)
static V3 background_bg(const Background& bg, V3 d) {
    double dz = std::fabs(0.0 * d.x + 0.0 * d.y + 1.0 * d.z);
    double t = rmin(std::sqrt(1.0 - dz * dz) / bg.scale, 1.0);
    return v3(lerp(t, bg.inner.x, bg.outer.x), lerp(t, bg.inner.y, bg.outer.y), lerp(t, bg.inner.z, bg.outer.z));
}

struct SampleAOV { uint32_t prim_id; double t; uint32_t occl_mask; bool unsupported; };

// Optional trace of one call tree of li() (orc_debug_li): every ray it casts, in order, as 8 doubles
// {kind (0 path ray, 1 shadow ray), depth, o.xyz, d.xyz} followed by {prim id or -1, t}.
static thread_local std::vector<double>* g_trace = nullptr;
static void trace_ray(int kind, uint32_t depth, const Ray& r, double prim, double t) {
    if (!g_trace) return;
    const double v[10] = {(double)kind, (double)depth, r.o.x, r.o.y, r.o.z, r.d.x, r.d.y, r.d.z, prim, t};
    g_trace->insert(g_trace->end(), v, v + 10);
}
// integrate/integrate.rs:23-132
static V3 li(const Accel& acc, const Ray& ray, uint32_t depth, SampleAOV* aov) {
    const Scene& sc = *acc.scene;
    if (g_cnt) { if (depth == 0) g_cnt->primary++; else g_cnt->secondary++; }
    RayIsect isect = isect_default();
    const Primitive* shape = acc.root->intersect(ray, isect);
    if (aov) { aov->prim_id = 0xFFFFFFFFu; aov->t = INF; aov->occl_mask = 0; aov->unsupported = false; }
    trace_ray(0, depth, ray, shape ? (double)isect.prim_id : -1.0, isect.t);
    if (!shape) return background_bg(sc.background, normalize(ray.d));
    if (g_cnt && depth == 0) g_cnt->primary_hits++;
    Material material;
    if (!shape->material(material)) material = isect.material;
    if (aov) { aov->prim_id = isect.prim_id; aov->t = isect.t; }
    SurfaceInteraction si = surface_from(ray, isect);
    V3 n = si.ns, wo = si.wo;
    V3 p = si.p + si.p_err;
    BSDF bsdf;
    if (!scattering(material, si, bsdf)) { if (aov) aov->unsupported = true; return v3(0, 0, 0); }
    V3 output = v3(0, 0, 0);
    for (size_t li_ = 0; li_ < sc.lights.size(); li_++) {
        const Light& light = sc.lights[li_];
        // light/point.rs:42-54
        Ray sray = ray_new(p, light.position - p);
        if (g_cnt) g_cnt->shadow++;
        RayIsect si2 = isect_default();
        const Primitive* blocker = acc.root->intersect(sray, si2);
        trace_ray(1, depth, sray, blocker ? (double)si2.prim_id : -1.0, si2.t);
        if (si2.t < 1.0) { if (g_cnt) g_cnt->shadow_occluded++; if (aov) aov->occl_mask |= (1u << li_); continue; }
        V3 wi = light.position - p;
        double d = magnitude(wi);
        double f_att = light.falloff[0] + light.falloff[1] * d + light.falloff[2] * d * d;
        if (f_att == 0.0) continue;
        wi = normalize(wi);
        double wi_dot_n = dot(wi, n);
        V3 f = bsdf.f(wo, wi);
        output = output + (mul_el(PI * light.intensity, f) * wi_dot_n / f_att);
    }
    output = output + mul_el(sc.ambient, bsdf.f(wo, n));
    V3 refracted = v3(0, 0, 0), reflected = v3(0, 0, 0);
    if (depth < sc.recursion) {                                           // integrate.rs:69-77
        {   // specular_transmit, integrate.rs:108-132
            LightSample s = bsdf.sample_f(wo, BX_TRANSMISSION | BX_SPECULAR);
            if (!(s.pdf <= 0.0 || is_zero(s.spectrum) || std::fabs(dot(s.wi, n)) == 0.0)) {
                Ray r = ray_new(si.p - si.p_err, s.wi);
                V3 l = li(acc, r, depth + 1, nullptr);
                refracted = mul_el(s.spectrum, l) * std::fabs(dot(s.wi, n)) / s.pdf;
            }
        }
        {   // specular_reflect, integrate.rs:82-106
            LightSample s = bsdf.sample_f(wo, BX_REFLECTION | BX_SPECULAR);
            if (!(s.pdf <= 0.0 || is_zero(s.spectrum) || dot(s.wi, n) <= 0.0)) {
                V3 wr = -1.0 * wo + 2.0 * dot(wo, n) * n;                 // bxdf::util::reflect, mod.rs:160-162
                Ray r = ray_new(si.p + si.p_err, wr);
                V3 l = li(acc, r, depth + 1, nullptr);
                reflected = mul_el(s.spectrum, l);
            }
        }
    }
    return output + reflected + refracted;                                // integrate.rs:79
}

// img.rs:65-67
static inline uint8_t to_byte(double c) {
    double v = std::round(rmin(rmax(c, 0.0), 1.0) * 255.0);
    if (!(v == v)) return 0;
    if (v <= 0.0) return 0;
    if (v >= 255.0) return 255;
    return (uint8_t)v;
}

// camera.rs:113-146
static void camera_sample(const Camera& c, uint32_t x, uint32_t y, uint32_t w, uint32_t h, std::vector<Ray>& rays) {
    double winv = 1.0 / (double)w, hinv = 1.0 / (double)h, aspect = (double)w / (double)h;   // film.rs:36-45
    double iph = c.image_plane_height;
    double ipw = iph * aspect;
    double pixel_size = iph * hinv;
    double sep = c.distance * pixel_size;
    double sox = ((double)x * winv - 0.5) * ipw;
    double soy = (0.5 - (double)(y + 1) * hinv) * iph;
    V3 origin = c.origin + (soy * c.pixel_separation * c.up) + (sox * c.pixel_separation * c.aux);
    V3 d = c.view + (soy * c.up) + (sox * c.aux);
    V3 updiff = c.up * sep, auxdiff = c.aux * sep;
    V3 halfdiff = updiff * 0.5 + auxdiff * 0.5;
    size_t dim = c.root;
    for (size_t i = 0; i < dim; i++)
        for (size_t j = 0; j < dim; j++) {
            double fi = (double)i, fj = (double)j;
            V3 dd = d + (fj * updiff) + (fi * auxdiff) + halfdiff;
            rays[i * dim + j] = ray_new(origin, dd);
        }
}

// lib.rs:110-162
static void capture_subset(const Accel& acc, size_t k, size_t n, uint32_t w, uint32_t h, uint8_t* rgba,
                           uint32_t* aov_id, double* aov_t, uint32_t* aov_occl, double* aov_li, Counters* cnt,
                           std::atomic<int>* unsupported) {
    const Scene& sc = *acc.scene;
    g_cnt = cnt;
    size_t area = (size_t)w * h;
    size_t spp = sc.camera.root * sc.camera.root;
    std::vector<Ray> rays(spp);
    double weight = 1.0 / (double)spp;
    for (size_t off = k; off < area; off += n) {
        uint32_t x = (uint32_t)(off % w), y = (uint32_t)(off / w);
        camera_sample(sc.camera, x, y, w, h, rays);
        V3 color = v3(0, 0, 0);
        for (size_t s = 0; s < spp; s++) {     // integrate.rs:16-20
            SampleAOV aov;
            bool want = aov_id || aov_t || aov_occl || unsupported;
            V3 c = li(acc, rays[s], 0, want ? &aov : nullptr);
            if (want && aov.unsupported && unsupported) unsupported->store(1);
            if (aov_id) aov_id[off * spp + s] = aov.prim_id;
            if (aov_t) aov_t[off * spp + s] = aov.t;
            if (aov_occl) aov_occl[off * spp + s] = aov.occl_mask;
            if (aov_li) { aov_li[(off * spp + s) * 3 + 0] = c.x; aov_li[(off * spp + s) * 3 + 1] = c.y; aov_li[(off * spp + s) * 3 + 2] = c.z; }
            color = color + c;
        }
        color = color * weight;
        uint8_t* px = rgba + off * 4;          // img.rs:46-61
        px[0] = to_byte(color.x); px[1] = to_byte(color.y); px[2] = to_byte(color.z); px[3] = 255;
    }
    g_cnt = nullptr;
}

}  // namespace orc

// ================================================================ C interface (ctypes)
using namespace orc;
extern "C" {

struct orc_counters {
    uint64_t node_tests, sphere_tests, cuboid_tests, tri_tests, primary, primary_hits, shadow, shadow_occluded, exact_ties;
};

void* orc_scene_new() { return new Scene(); }
void orc_scene_free(void* s) { delete (Scene*)s; }
static Material mk_mat(int kind, const double* kd, const double* ks, double rough, double rough2) {
    return Material{kind, v3(kd[0], kd[1], kd[2]), v3(ks[0], ks[1], ks[2]), rough, rough2};
}
void orc_set_max_recursion_depth(void* s, uint32_t depth) { ((Scene*)s)->recursion = depth; }          // scene.rs
void orc_set_perspective_camera(void* s, double fov) { ((Scene*)s)->camera.reset(true, fov); }
void orc_set_orthographic_camera(void* s, double height) { ((Scene*)s)->camera.reset(false, height); }
void orc_look_at(void* s, const double* o, const double* l, const double* u) {
    ((Scene*)s)->camera.look_at(v3(o[0], o[1], o[2]), v3(l[0], l[1], l[2]), v3(u[0], u[1], u[2]));
}
void orc_set_supersampling(void* s, int base) { ((Scene*)s)->camera.set_supersampling((uint8_t)base); }
void orc_set_ambient_light(void* s, const double* c) { ((Scene*)s)->ambient = v3(c[0], c[1], c[2]); }
void orc_set_radial_background(void* s, const double* in, const double* out, double scale) {
    ((Scene*)s)->background = Background{v3(in[0], in[1], in[2]), v3(out[0], out[1], out[2]), scale};
}
void orc_add_point_light(void* s, const double* p, const double* i, const double* f) {
    ((Scene*)s)->lights.push_back(Light{v3(p[0], p[1], p[2]), v3(i[0], i[1], i[2]), {f[0], f[1], f[2]}});
}
int orc_add_mesh(void* s, const float* pos, uint64_t nv, const uint32_t* vi, uint64_t ntri,
                 const float* nrm, uint64_t nn, const uint32_t* ni) {
    Scene* sc = (Scene*)s;
    Mesh m;
    m.pos.assign(pos, pos + 3 * nv);
    m.vi.assign(vi, vi + 3 * ntri);
    if (nrm && nn) { m.nrm.assign(nrm, nrm + 3 * nn); m.ni.assign(ni, ni + 3 * ntri); }
    sc->meshes.push_back(std::move(m));
    return (int)sc->meshes.size() - 1;
}
int orc_agg_new(void* s) { Scene* sc = (Scene*)s; sc->aggs.emplace_back(); return (int)sc->aggs.size() - 1; }
void orc_agg_add_sphere(void* s, int ag, const double* c, double r, int kind, const double* kd, const double* ks, double rough, double rough2) {
    ((Scene*)s)->aggs[ag].contents.push_back(SceneNode{N_SPHERE, v3(c[0], c[1], c[2]), v3(0, 0, 0), r, mk_mat(kind, kd, ks, rough, rough2), true, -1});
}
void orc_agg_add_spheres(void* s, int ag, uint64_t n, const double* c, const double* r, int nmat, const int* kinds,
                         const double* kd, const double* ks, const double* rough, const double* rough2, const int* mat_index) {
    Aggregate& a = ((Scene*)s)->aggs[ag];
    a.contents.reserve(a.contents.size() + n);
    for (uint64_t i = 0; i < n; i++) {
        int m = mat_index[i]; (void)nmat;
        a.contents.push_back(SceneNode{N_SPHERE, v3(c[3 * i], c[3 * i + 1], c[3 * i + 2]), v3(0, 0, 0), r[i],
                                       mk_mat(kinds[m], kd + 3 * m, ks + 3 * m, rough[m], rough2[m]), true, -1});
    }
}
void orc_agg_add_cube(void* s, int ag, const double* o, double dim, int kind, const double* kd, const double* ks, double rough, double rough2) {
    ((Scene*)s)->aggs[ag].contents.push_back(SceneNode{N_CUBE, v3(o[0], o[1], o[2]), v3(0, 0, 0), dim, mk_mat(kind, kd, ks, rough, rough2), true, -1});
}
void orc_agg_add_box(void* s, int ag, const double* a, const double* b, int kind, const double* kd, const double* ks, double rough, double rough2) {
    ((Scene*)s)->aggs[ag].contents.push_back(SceneNode{N_CUBOID, v3(a[0], a[1], a[2]), v3(b[0], b[1], b[2]), 0.0, mk_mat(kind, kd, ks, rough, rough2), true, -1});
}
void orc_agg_add_mesh(void* s, int ag, int mesh, int has_mat, int kind, const double* kd, const double* ks, double rough, double rough2) {
    ((Scene*)s)->aggs[ag].contents.push_back(SceneNode{N_MESH, v3(0, 0, 0), v3(0, 0, 0), 0.0, mk_mat(kind, kd, ks, rough, rough2), has_mat != 0, mesh});
}
void orc_agg_add_group(void* s, int ag, int child) {
    ((Scene*)s)->aggs[ag].contents.push_back(SceneNode{N_GROUP, v3(0, 0, 0), v3(0, 0, 0), 0.0, mat_default(), false, child});
}
void orc_agg_swap_backface(void* s, int ag) { Aggregate& a = ((Scene*)s)->aggs[ag]; a.swap_backface = !a.swap_backface; }
void orc_agg_translate(void* s, int ag, const double* d) { ((Scene*)s)->aggs[ag].transform.concat_self(t_translate(v3(d[0], d[1], d[2]))); }
void orc_agg_scale(void* s, int ag, double x, double y, double z) { ((Scene*)s)->aggs[ag].transform.concat_self(t_scale(x, y, z)); }
void orc_agg_rotate_axis(void* s, int ag, int axis, double deg) { ((Scene*)s)->aggs[ag].transform.concat_self(t_rotate_axis(axis, deg)); }
void orc_agg_rotate(void* s, int ag, double deg, const double* a) { ((Scene*)s)->aggs[ag].transform.concat_self(t_rotate(deg, v3(a[0], a[1], a[2]))); }

// Accel::from (lib.rs:42, bvh.rs:135).  Returns NULL where the reference would not terminate (Q9/Q10).
void* orc_accel_build(void* s) {
    auto t0 = std::chrono::steady_clock::now();
    Accel* a = new Accel();
    a->scene = (Scene*)s;
    a->root = a->from_aggregate(0);
    if (a->failed) { delete a; return nullptr; }
    a->build_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    return a;
}
void orc_accel_free(void* a) { delete (Accel*)a; }
double orc_accel_build_ms(void* a) { return ((Accel*)a)->build_ms; }
uint32_t orc_accel_prim_count(void* a) { return ((Accel*)a)->next_id; }

// Introspection of one BVH level for builder parity tests.  `path` walks nested
// BVH primitives: path[i] is the primitive index inside the current level.
static const BVH* walk(const Accel* a, const int* path, int npath) {
    const BVH* b = a->root.get();
    for (int i = 0; i < npath; i++) {
        b = dynamic_cast<const BVH*>(b->primitives[path[i]].get());
        if (!b) return nullptr;
    }
    return b;
}
int64_t orc_bvh_node_count(void* a, const int* path, int npath) { const BVH* b = walk((Accel*)a, path, npath); return b ? (int64_t)b->nodes.size() : -1; }
int64_t orc_bvh_prim_count(void* a, const int* path, int npath) { const BVH* b = walk((Accel*)a, path, npath); return b ? (int64_t)b->primitives.size() : -1; }
// nodes: bounds[6] doubles, meta[3] u32 (leaf, a, b) per node; order: u64 per primitive
int orc_bvh_dump(void* a, const int* path, int npath, double* bounds, uint32_t* meta, uint64_t* order) {
    const BVH* b = walk((Accel*)a, path, npath);
    if (!b) return -1;
    for (size_t i = 0; i < b->nodes.size(); i++) {
        const LinearNode& n = b->nodes[i];
        bounds[6 * i + 0] = n.bounds.mn.x; bounds[6 * i + 1] = n.bounds.mn.y; bounds[6 * i + 2] = n.bounds.mn.z;
        bounds[6 * i + 3] = n.bounds.mx.x; bounds[6 * i + 4] = n.bounds.mx.y; bounds[6 * i + 5] = n.bounds.mx.z;
        meta[3 * i + 0] = n.leaf ? 1u : 0u; meta[3 * i + 1] = n.a; meta[3 * i + 2] = n.b;
    }
    for (size_t i = 0; i < b->order.size(); i++) order[i] = (uint64_t)b->order[i];
    return 0;
}

// capture (lib.rs:55-104) with `threads` workers (0 = hardware_concurrency), or only the
// subsets [k0, k0 + kcount) of n when kcount > 0 (capture_subset, lib.rs:110).
// Optional outputs may be NULL.  Returns 0, or 1 if a material outside the path was hit,
// or 2 on traversal stack overflow (the reference would panic).
int orc_capture(void* accel, uint32_t w, uint32_t h, int threads, uint64_t n, uint64_t k0, uint64_t kcount,
                uint8_t* rgba, uint32_t* aov_id, double* aov_t, uint32_t* aov_occl, double* aov_li,
                orc_counters* counters, double* render_ms) {
    Accel* acc = (Accel*)accel;
    size_t nthreads = threads > 0 ? (size_t)threads : std::max<size_t>(1, std::thread::hardware_concurrency());
    std::atomic<int> unsupported{0};
    auto t0 = std::chrono::steady_clock::now();
    std::vector<Counters> cnts(nthreads);
    std::vector<std::thread> th;
    if (kcount == 0) {            // full capture: barrel k of n = nthreads
        for (size_t k = 1; k < nthreads; k++)
            th.emplace_back([&, k] { capture_subset(*acc, k, nthreads, w, h, rgba, aov_id, aov_t, aov_occl, aov_li, counters ? &cnts[k] : nullptr, &unsupported); });
        capture_subset(*acc, 0, nthreads, w, h, rgba, aov_id, aov_t, aov_occl, aov_li, counters ? &cnts[0] : nullptr, &unsupported);
    } else {                      // explicit subsets, distributed over the workers
        std::atomic<uint64_t> next{0};
        auto work = [&](size_t tid) {
            for (;;) {
                uint64_t i = next.fetch_add(1);
                if (i >= kcount) break;
                capture_subset(*acc, (size_t)(k0 + i), (size_t)n, w, h, rgba, aov_id, aov_t, aov_occl, aov_li, counters ? &cnts[tid] : nullptr, &unsupported);
            }
        };
        for (size_t k = 1; k < nthreads; k++) th.emplace_back(work, k);
        work(0);
    }
    for (auto& t : th) t.join();
    if (render_ms) *render_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    if (counters) {
        Counters tot; for (auto& c : cnts) tot.add(c);
        *counters = orc_counters{tot.node_tests, tot.sphere_tests, tot.cuboid_tests, tot.tri_tests, tot.primary,
                                 tot.primary_hits, tot.shadow, tot.shadow_occluded, tot.exact_ties};
    }
    // stack overflow flags
    std::vector<const BVH*> st{acc->root.get()};
    bool overflow = false;
    while (!st.empty()) {
        const BVH* b = st.back(); st.pop_back();
        if (b->stack_overflow.load()) overflow = true;
        for (auto& p : b->primitives) if (auto c = dynamic_cast<const BVH*>(p.get())) st.push_back(c);
    }
    if (overflow) return 2;
    return unsupported.load() ? 1 : 0;
}

// ---- single-primitive entry points for the reference's unit-test vectors (SURVEY §4)
// out: t, ng[3] (RayIntersection::ng, not face-forwarded), ns[3]; returns 1 on hit.
static int finish(bool hit, const RayIsect& is, double* out) {
    out[0] = is.t;
    if (hit) { V3 g = isect_ng(is), s = isect_ns(is); out[1] = g.x; out[2] = g.y; out[3] = g.z; out[4] = s.x; out[5] = s.y; out[6] = s.z; }
    return hit ? 1 : 0;
}
int orc_test_sphere(const double* c, double r, const double* o, const double* d, double* out) {
    Sphere s; s.origin = v3(c[0], c[1], c[2]); s.radius = r; s.mat = mat_default(); s.id = 0;
    RayIsect is = isect_default();
    bool hit = s.intersect(ray_new(v3(o[0], o[1], o[2]), v3(d[0], d[1], d[2])), is) != nullptr;
    return finish(hit, is, out);
}
int orc_test_cuboid(const double* mn, const double* mx, const double* o, const double* d, double* out) {
    Cuboid c; c.bounds = b_new(v3(mn[0], mn[1], mn[2]), v3(mx[0], mx[1], mx[2])); c.mat = mat_default(); c.id = 0;
    RayIsect is = isect_default();
    bool hit = c.intersect(ray_new(v3(o[0], o[1], o[2]), v3(d[0], d[1], d[2])), is) != nullptr;
    return finish(hit, is, out);
}
// All triangles of a mesh tested in TriangleIterator order against one record (triangle.rs:411-431).
int orc_test_mesh(const float* pos, uint64_t nv, const uint32_t* vi, uint64_t ntri, const float* nrm, uint64_t nn,
                  const uint32_t* ni, const double* o, const double* d, double* out, int64_t* which) {
    Mesh m; m.pos.assign(pos, pos + 3 * nv); m.vi.assign(vi, vi + 3 * ntri);
    if (nrm && nn) { m.nrm.assign(nrm, nrm + 3 * nn); m.ni.assign(ni, ni + 3 * ntri); }
    RayIsect is = isect_default(); bool hit = false; *which = -1;
    Ray ray = ray_new(v3(o[0], o[1], o[2]), v3(d[0], d[1], d[2]));
    for (uint64_t i = 0; i < ntri; i++) {
        Triangle t; t.mesh = &m; t.tri = (uint32_t)i; t.id = (uint32_t)i;
        if (t.intersect(ray, is)) { hit = true; *which = (int64_t)i; }
    }
    return finish(hit, is, out);
}
// surface.rs:194-200: SurfaceInteraction::from on a hand-made record; out = ng[3]
void orc_test_surface(double t, const double* dpdu, const double* dpdv, const double* o, const double* d, double* out) {
    RayIsect is = isect_new(t, v3(dpdu[0], dpdu[1], dpdu[2]), v3(dpdv[0], dpdv[1], dpdv[2]));
    SurfaceInteraction si = surface_from(ray_new(v3(o[0], o[1], o[2]), v3(d[0], d[1], d[2])), is);
    out[0] = si.ng.x; out[1] = si.ng.y; out[2] = si.ng.z;
}
// Substance::evaluate (fresnel.rs:22-33).  kind 0 dielectric (p = eta_i, eta_t), 1 conductor (p = eta_i[3], eta_t[3], k[3]), 2 no-op.
void orc_test_fresnel(int kind, double cos_i, const double* p, double* out) {
    Substance s; s.kind = kind;
    if (kind == SUB_DIELECTRIC) { s.eta_i = p[0]; s.eta_t = p[1]; }
    if (kind == SUB_CONDUCTOR) { s.c_eta_i = v3(p[0], p[1], p[2]); s.c_eta_t = v3(p[3], p[4], p[5]); s.c_k = v3(p[6], p[7], p[8]); }
    V3 f = s.evaluate(cos_i); out[0] = f.x; out[1] = f.y; out[2] = f.z;
}
// Material::scattering on a hand-made interaction (ng, ns, normalised dpdu), then BSDF::f(wo, wi) and the two Whitted samples
// (bsdf.rs:73-140): out_f[3]; out_refl = spectrum[3], wi[3], pdf; out_trans likewise.
void orc_test_bsdf(int kind, const double* kd, const double* ks, double rough, double rough2, const double* frame,
                   const double* wo, const double* wi, double* out_f, double* out_refl, double* out_trans) {
    SurfaceInteraction si;
    si.ng = v3(frame[0], frame[1], frame[2]); si.ns = v3(frame[3], frame[4], frame[5]); si.s_dpdu = v3(frame[6], frame[7], frame[8]);
    BSDF b;
    scattering(mk_mat(kind, kd, ks, rough, rough2), si, b);
    V3 o = v3(wo[0], wo[1], wo[2]), i = v3(wi[0], wi[1], wi[2]);
    V3 f = b.f(o, i); out_f[0] = f.x; out_f[1] = f.y; out_f[2] = f.z;
    LightSample r = b.sample_f(o, BX_REFLECTION | BX_SPECULAR), t = b.sample_f(o, BX_TRANSMISSION | BX_SPECULAR);
    double* dst[2] = {out_refl, out_trans}; const LightSample* src[2] = {&r, &t};
    for (int k = 0; k < 2; k++) {
        dst[k][0] = src[k]->spectrum.x; dst[k][1] = src[k]->spectrum.y; dst[k][2] = src[k]->spectrum.z;
        dst[k][3] = src[k]->wi.x; dst[k][4] = src[k]->wi.y; dst[k][5] = src[k]->wi.z; dst[k][6] = src[k]->pdf;
    }
}
// Exact f64 re-test of ONE canonical primitive against one ray (SURVEY Appendix E step 1):
// returns t or +inf.  The primitive is located by canonical id through the accel.
double orc_retest_prim(void* accel, uint32_t prim_id, const double* o, const double* d) {
    Accel* acc = (Accel*)accel;
    Ray world = ray_new(v3(o[0], o[1], o[2]), v3(d[0], d[1], d[2]));
    // every nested level sees the ray through its own inverse transform, applied level by level (bvh.rs:462)
    std::vector<std::pair<const BVH*, Ray>> st;
    st.push_back({acc->root.get(), ray_new(m4_point(acc->root->transform.minv, world.o), m4_vector(acc->root->transform.minv, world.d))});
    while (!st.empty()) {
        const BVH* b = st.back().first; const Ray ray = st.back().second; st.pop_back();
        for (auto& p : b->primitives) {
            if (auto c = dynamic_cast<const BVH*>(p.get())) {
                st.push_back({c, ray_new(m4_point(c->transform.minv, ray.o), m4_vector(c->transform.minv, ray.d))});
                continue;
            }
            uint32_t id = 0xFFFFFFFFu;
            if (auto s = dynamic_cast<const Sphere*>(p.get())) id = s->id;
            else if (auto c2 = dynamic_cast<const Cuboid*>(p.get())) id = c2->id;
            else if (auto t = dynamic_cast<const Triangle*>(p.get())) id = t->id;
            if (id == prim_id) { RayIsect is = isect_default(); return p->intersect(ray, is) ? is.t : INF; }
        }
    }
    return INF;
}
// Closest hit of caller-supplied rays (Accel::intersect, bvh.rs:461-522): ids = canonical primitive id or 0xFFFFFFFF, t = isect.t.
// ng / ns (3 doubles per ray, NULL = not wanted): RayIntersection::ng() / ns() (surface.rs:107-118) of the world-space record the
// root returns, i.e. after transform_isect and the swap_backface flips of every level; zeros on a miss.
void orc_trace_rays(void* accel, const double* rays, uint64_t n, uint32_t* ids, double* ts, double* ng, double* ns) {
    Accel* acc = (Accel*)accel;
    for (uint64_t i = 0; i < n; i++) {
        Ray r = ray_new(v3(rays[6 * i], rays[6 * i + 1], rays[6 * i + 2]), v3(rays[6 * i + 3], rays[6 * i + 4], rays[6 * i + 5]));
        RayIsect is = isect_default();
        const Primitive* shape = acc->root->intersect(r, is);
        ids[i] = shape ? is.prim_id : 0xFFFFFFFFu;
        ts[i] = shape ? is.t : INF;
        const V3 g = shape ? isect_ng(is) : v3(0, 0, 0), s = shape ? isect_ns(is) : v3(0, 0, 0);
        if (ng) { ng[3 * i] = g.x; ng[3 * i + 1] = g.y; ng[3 * i + 2] = g.z; }
        if (ns) { ns[3 * i] = s.x; ns[3 * i + 1] = s.y; ns[3 * i + 2] = s.z; }
    }
}
// li() of one ray with a trace of every ray cast below it (10 doubles each, see trace_ray); returns the number of rays, out_li = radiance.
uint64_t orc_debug_li(void* accel, const double* ray, double* out_li, double* out_trace, uint64_t cap) {
    Accel* acc = (Accel*)accel;
    std::vector<double> tr;
    g_trace = &tr;
    V3 c = li(*acc, ray_new(v3(ray[0], ray[1], ray[2]), v3(ray[3], ray[4], ray[5])), 0, nullptr);
    g_trace = nullptr;
    out_li[0] = c.x; out_li[1] = c.y; out_li[2] = c.z;
    const uint64_t n = tr.size() / 10;
    for (uint64_t i = 0; i < n && i < cap; i++) for (int k = 0; k < 10; k++) out_trace[10 * i + k] = tr[10 * i + k];
    return n;
}
// Camera rays for one pixel (camera.rs:113-146): out = spp * 6 doubles (origin, d)
void orc_camera_sample(void* s, uint32_t x, uint32_t y, uint32_t w, uint32_t h, double* out) {
    Scene* sc = (Scene*)s;
    std::vector<Ray> rays(sc->camera.root * sc->camera.root);
    camera_sample(sc->camera, x, y, w, h, rays);
    for (size_t i = 0; i < rays.size(); i++) {
        out[6 * i + 0] = rays[i].o.x; out[6 * i + 1] = rays[i].o.y; out[6 * i + 2] = rays[i].o.z;
        out[6 * i + 3] = rays[i].d.x; out[6 * i + 4] = rays[i].d.y; out[6 * i + 5] = rays[i].d.z;
    }
}
int orc_hardware_threads() { return (int)std::max<size_t>(1, std::thread::hardware_concurrency()); }

}  // extern "C"
