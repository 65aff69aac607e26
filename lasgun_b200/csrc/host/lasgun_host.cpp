// Host side above the C ABI: scene builder mirror, HLBVH build (the reference's algorithm,
// src/accelerators/bvh.rs:135-453), flattening into lgb_scene_desc arrays, capture.
// Product code: does not include or link anything under oracle/.
#include "../../../include/lasgun_host.hpp"

#include "../lgb_parallel.hpp"

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <mutex>

namespace lasgun {

static const double kPi = 3.14159265358979323846264338327950288;

// ------------------------------------------------------------------ materials, camera, film
Material Material::matte(const double kd[3], double sigma) {
    Material m; m.kind = Matte; for (int i = 0; i < 3; i++) { m.kd[i] = kd[i]; m.ks[i] = 0.0; }
    m.roughness = std::min(std::max(sigma, 0.0), 90.0);      // matte.rs:14-16
    return m;
}
Material Material::plastic(const double kd[3], const double ks[3], double roughness) {
    Material m; m.kind = Plastic; for (int i = 0; i < 3; i++) { m.kd[i] = kd[i]; m.ks[i] = ks[i]; }
    m.roughness = roughness;
    return m;
}

Material Material::metal(const double eta[3], const double k[3], double u_roughness, double v_roughness) {   // mod.rs:30-34
    Material m; m.kind = Metal; for (int i = 0; i < 3; i++) { m.kd[i] = eta[i]; m.ks[i] = k[i]; }
    m.roughness = u_roughness; m.roughness_v = v_roughness;
    return m;
}
Material Material::glass(const double kr[3], const double kt[3], double eta) {                                // mod.rs:36-41
    Material m; m.kind = Glass; for (int i = 0; i < 3; i++) { m.kd[i] = kr[i]; m.ks[i] = kt[i]; }
    m.roughness = eta;
    return m;
}
Material Material::mirror(const double kr[3]) {                                                              // mod.rs:43-46
    Material m; m.kind = Mirror; for (int i = 0; i < 3; i++) { m.kd[i] = kr[i]; m.ks[i] = 0.0; }
    return m;
}

double Camera::plane_height(double focal) const {              // camera.rs:158-164
    return is_perspective ? focal * std::tan(param * kPi / 360.0) * 2.0 : param;
}
Camera Camera::perspective(double fov) {
    Camera c; c.is_perspective = true; c.param = fov;
    c.image_plane_height = c.plane_height(1.0); c.pixel_separation = 0.0;
    return c;
}
Camera Camera::orthographic(double height) {
    Camera c; c.is_perspective = false; c.param = height;
    c.image_plane_height = c.plane_height(1.0); c.pixel_separation = 1.0;
    return c;
}
static inline void cross3(const double a[3], const double b[3], double o[3]) {
    o[0] = a[1] * b[2] - a[2] * b[1]; o[1] = a[2] * b[0] - a[0] * b[2]; o[2] = a[0] * b[1] - a[1] * b[0];
}
static inline double dot3(const double a[3], const double b[3]) { return a[0] * b[0] + a[1] * b[1] + a[2] * b[2]; }
static inline void normalize3(double v[3]) { double s = 1.0 / std::sqrt(dot3(v, v)); v[0] *= s; v[1] *= s; v[2] *= s; }
void Camera::look_at(const double o[3], const double look[3], const double upv[3]) {   // camera.rs:85-94
    double v[3] = {look[0] - o[0], look[1] - o[1], look[2] - o[2]};
    double ax[3]; cross3(v, upv, ax);
    double u[3]; cross3(ax, v, u);
    normalize3(u); normalize3(ax);
    for (int i = 0; i < 3; i++) { origin[i] = o[i]; up[i] = u[i]; aux[i] = ax[i]; view[i] = v[i]; }
    image_plane_height = plane_height(std::sqrt(dot3(v, v)));
}
void Camera::set_supersampling(uint8_t base) {                  // camera.rs:189-193
    if (base == 255) throw Error(LGB_ERR_INVALID, "set_supersampling: base must be < 255");
    root = (size_t)base + 1; distance = 1.0 / (double)root;
}

Film::Film(uint32_t width, uint32_t height)
    : w(width), h(height), winv(1.0 / width), hinv(1.0 / height), aspect((double)width / (double)height),
      own((size_t)width * height * 4, 0), ptr(own.data()) {}
Film::Film(uint32_t width, uint32_t height, uint8_t* external)
    : w(width), h(height), winv(1.0 / width), hinv(1.0 / height), aspect((double)width / (double)height), ptr(external) {}

// ------------------------------------------------------------------ transforms (cgmath column-major)
Transform::Transform() {
    for (int i = 0; i < 16; i++) m[i] = minv[i] = (i % 5 == 0) ? 1.0 : 0.0;
}
static void mat_mul(const double a[16], const double b[16], double o[16]) {
    double r[16];
    for (int c = 0; c < 4; c++)
        for (int rr = 0; rr < 4; rr++)
            r[4 * c + rr] = a[0 + rr] * b[4 * c] + a[4 + rr] * b[4 * c + 1] + a[8 + rr] * b[4 * c + 2] + a[12 + rr] * b[4 * c + 3];
    std::memcpy(o, r, sizeof r);
}
static void concat_self(Transform& t, const double om[16], const double ominv[16]) {   // transform.rs:191-197
    double nm[16], nminv[16];
    mat_mul(om, t.m, nm); mat_mul(t.minv, ominv, nminv);
    std::memcpy(t.m, nm, sizeof nm); std::memcpy(t.minv, nminv, sizeof nminv);
    t.identity = false;
}
static void transpose(const double a[16], double o[16]) { for (int c = 0; c < 4; c++) for (int r = 0; r < 4; r++) o[4 * c + r] = a[4 * r + c]; }
Aggregate& Aggregate::translate(const double d[3]) {
    Transform a, b; a.m[12] = d[0]; a.m[13] = d[1]; a.m[14] = d[2]; b.m[12] = -d[0]; b.m[13] = -d[1]; b.m[14] = -d[2];
    concat_self(transform, a.m, b.m); return *this;
}
Aggregate& Aggregate::scale(double x, double y, double z) {
    Transform a, b; a.m[0] = x; a.m[5] = y; a.m[10] = z; b.m[0] = 1.0 / x; b.m[5] = 1.0 / y; b.m[10] = 1.0 / z;
    concat_self(transform, a.m, b.m); return *this;
}
static Aggregate& rotate_axis(Aggregate& g, int axis, double deg) {
    double th = deg * kPi / 180.0, s = std::sin(th), c = std::cos(th);
    Transform a;
    if (axis == 0) { a.m[5] = c; a.m[6] = s; a.m[9] = -s; a.m[10] = c; }
    else if (axis == 1) { a.m[0] = c; a.m[2] = -s; a.m[8] = s; a.m[10] = c; }
    else { a.m[0] = c; a.m[1] = s; a.m[4] = -s; a.m[5] = c; }
    double inv[16]; transpose(a.m, inv);
    concat_self(g.transform, a.m, inv); return g;
}
Aggregate& Aggregate::rotate_x(double t) { return rotate_axis(*this, 0, t); }
Aggregate& Aggregate::rotate_y(double t) { return rotate_axis(*this, 1, t); }
Aggregate& Aggregate::rotate_z(double t) { return rotate_axis(*this, 2, t); }
Aggregate& Aggregate::rotate(double deg, const double ax[3]) {
    double th = deg * kPi / 180.0, s = std::sin(th), c = std::cos(th), k = 1.0 - c;
    Transform a;
    a.m[0] = k * ax[0] * ax[0] + c;         a.m[1] = k * ax[0] * ax[1] + s * ax[2]; a.m[2] = k * ax[0] * ax[2] - s * ax[1];
    a.m[4] = k * ax[0] * ax[1] - s * ax[2]; a.m[5] = k * ax[1] * ax[1] + c;         a.m[6] = k * ax[1] * ax[2] + s * ax[0];
    a.m[8] = k * ax[0] * ax[2] + s * ax[1]; a.m[9] = k * ax[1] * ax[2] - s * ax[0]; a.m[10] = k * ax[2] * ax[2] + c;
    double inv[16]; transpose(a.m, inv);
    concat_self(transform, a.m, inv); return *this;
}

// ------------------------------------------------------------------ scene builder
static Aggregate::Node mk_node(Aggregate::Node::Kind k) {
    Aggregate::Node n; n.kind = k; n.r = 0.0; n.has_mat = false; n.ref = 0;
    for (int i = 0; i < 3; i++) n.a[i] = n.b[i] = 0.0;
    return n;
}
void Aggregate::add_group(Aggregate g) { Node n = mk_node(Node::Group); n.ref = groups.size(); groups.push_back(std::move(g)); contents.push_back(n); }
void Aggregate::add_sphere(const double c[3], double r, const Material& m) {
    Node n = mk_node(Node::Sphere); for (int i = 0; i < 3; i++) n.a[i] = c[i]; n.r = r; n.mat = m; n.has_mat = true; contents.push_back(n);
}
void Aggregate::add_cube(const double o[3], double dim, const Material& m) {
    Node n = mk_node(Node::Cube); for (int i = 0; i < 3; i++) n.a[i] = o[i]; n.r = dim; n.mat = m; n.has_mat = true; contents.push_back(n);
}
void Aggregate::add_box(const double a[3], const double b[3], const Material& m) {
    Node n = mk_node(Node::Cuboid); for (int i = 0; i < 3; i++) { n.a[i] = a[i]; n.b[i] = b[i]; } n.mat = m; n.has_mat = true; contents.push_back(n);
}
void Aggregate::add_obj(ObjRef mesh) { Node n = mk_node(Node::Mesh); n.ref = mesh.index; contents.push_back(n); }
void Aggregate::add_obj_of(ObjRef mesh, const Material& m) { Node n = mk_node(Node::Mesh); n.ref = mesh.index; n.mat = m; n.has_mat = true; contents.push_back(n); }

void Scene::set_solid_background(const double c[3]) { for (int i = 0; i < 3; i++) bg_inner[i] = bg_outer[i] = c[i]; bg_scale = 1.0; }
void Scene::set_radial_background(const double in[3], const double out[3], double scale) {
    for (int i = 0; i < 3; i++) { bg_inner[i] = in[i]; bg_outer[i] = out[i]; } bg_scale = scale;
}
void Scene::set_ambient_light(const double c[3]) { for (int i = 0; i < 3; i++) ambient[i] = c[i]; }
void Scene::add_point_light(const double p[3], const double in[3], const double f[3]) {
    Light l; for (int i = 0; i < 3; i++) { l.position[i] = p[i]; l.intensity[i] = in[i]; l.falloff[i] = f[i]; } lights.push_back(l);
}
ObjRef Scene::add_obj(ObjData mesh) {                            // scene.rs:109-115
    if (!smoothing) { mesh.normals.clear(); mesh.normal_faces.clear(); }
    if (mesh.faces.size() % 3 || mesh.positions.size() % 3) throw Error(LGB_ERR_INVALID, "add_obj: malformed mesh arrays");
    if (!mesh.normals.empty() && mesh.normal_faces.size() != mesh.faces.size()) throw Error(LGB_ERR_INVALID, "add_obj: normal_faces must match faces");
    for (uint32_t v : mesh.faces) if ((size_t)v * 3 >= mesh.positions.size()) throw Error(LGB_ERR_INVALID, "add_obj: face index out of range");
    for (uint32_t v : mesh.normal_faces) if ((size_t)v * 3 >= mesh.normals.size()) throw Error(LGB_ERR_INVALID, "add_obj: normal index out of range");
    meshes.push_back(std::move(mesh));
    return ObjRef{meshes.size() - 1};
}

// ------------------------------------------------------------------ HLBVH build of one level
namespace {

const double F64MAX = std::numeric_limits<double>::max();
struct Box {
    double mn[3], mx[3];
    static Box none() { Box b; for (int i = 0; i < 3; i++) { b.mn[i] = F64MAX; b.mx[i] = -F64MAX; } return b; }   // bounds.rs:152-157
    void grow(const Box& o) { for (int i = 0; i < 3; i++) { if (o.mn[i] < mn[i]) mn[i] = o.mn[i]; if (mx[i] < o.mx[i]) mx[i] = o.mx[i]; } }
    void grow_pt(const double p[3]) { for (int i = 0; i < 3; i++) { if (p[i] < mn[i]) mn[i] = p[i]; if (mx[i] < p[i]) mx[i] = p[i]; } }
    double area() const {                                                                                           // bounds.rs:110-114
        double d0 = mx[0] - mn[0], d1 = mx[1] - mn[1], d2 = mx[2] - mn[2];
        double half = d0 * d1 + d0 * d2 + d1 * d2;
        return half + half;
    }
};
inline uint32_t sat_u32(double v) { if (!(v == v) || v <= 0.0) return 0; if (v >= 4294967295.0) return 4294967295u; return (uint32_t)v; }
inline uint32_t spread10(uint32_t x) {                          // bvh.rs:590-598
    if (x == 1024u) x = 1023u;
    x = (x | (x << 16)) & 0x030000FFu;
    x = (x | (x << 8)) & 0x0300F00Fu;
    x = (x | (x << 4)) & 0x030C30C3u;
    x = (x | (x << 2)) & 0x09249249u;
    return x;
}

struct BuildNode { Box box; int left = -1, right = -1; uint32_t first = 0, count = 0; uint8_t axis = 0; };

// One BVH level (BVHAccel::new, bvh.rs:164-202).  `boxes[i]` is primitive i's bound.
struct LevelTree {
    std::vector<BuildNode> nodes;
    raw_vector<uint32_t> order;       // bvh.rs:56-59
    int root = -1;
    size_t total_nodes = 0;

    void build(const raw_vector<Box>& boxes, size_t per_node) {
        const size_t n = boxes.size();
        if (n == 0) throw Error(LGB_ERR_INVALID, "empty aggregate: the reference's BVH build does not terminate (bvh.rs:240,355-356)");
        const size_t max_prims = std::min<size_t>(per_node, 255);
        lgb::Pool& pool = lgb::Pool::get();
        order.resize(n);             // every slot is written exactly once by the treelet emission below
        // scene bounds (bvh.rs:212-213): min / max folds are order-independent, so the chunks may run in parallel
        Box bounds = Box::none();
        {
            const size_t nc = pool.chunks_of(n, 1 << 14);
            std::vector<Box> part(nc, Box::none());
            pool.for_range(n, 1 << 14, [&](size_t b, size_t e, size_t c) { for (size_t i = b; i < e; i++) part[c].grow(boxes[i]); });
            for (const Box& b : part) bounds.grow(b);
        }
        // Morton codes (bvh.rs:217-224, 575-579: z, y, z)
        raw_vector<uint32_t> code(n), idx(n), code2(n), idx2(n);
        pool.for_range(n, 1 << 14, [&](size_t b, size_t e, size_t) {
            for (size_t i = b; i < e; i++) {
                double off[3];
                for (int k = 0; k < 3; k++) {
                    double c = 0.5 * boxes[i].mn[k] + 0.5 * boxes[i].mx[k];        // bvh.rs:530
                    double o = c - bounds.mn[k];
                    if (bounds.mx[k] > bounds.mn[k]) o /= bounds.mx[k] - bounds.mn[k];   // bounds.rs:133-139
                    off[k] = o * 1024.0;
                }
                uint32_t z = spread10(sat_u32(off[2])), y = spread10(sat_u32(off[1]));
                code[i] = (z << 2) | (y << 1) | z;
                idx[i] = (uint32_t)i;
            }
        });
        // Stable LSD radix sort on the 30-bit key: the same permutation as the reference's 5 x 6-bit passes
        // (bvh.rs:600-635), three 10-bit passes with per-chunk histograms so that every pass is parallel and stable.
        {
            const size_t nc = std::max<size_t>(1, pool.chunks_of(n, 1 << 15));
            const size_t per = (n + nc - 1) / nc;
            std::vector<uint32_t> hist(nc * 1024);
            for (int pass = 0; pass < 3; pass++) {
                const int shift = 10 * pass;
                pool.run(nc, [&](size_t c) {
                    uint32_t* h = hist.data() + c * 1024; std::fill(h, h + 1024, 0u);
                    const size_t b = c * per, e = std::min(n, b + per);
                    for (size_t i = b; i < e; i++) h[(code[i] >> shift) & 1023u]++;
                });
                uint32_t run = 0;
                for (int d = 0; d < 1024; d++) for (size_t c = 0; c < nc; c++) { uint32_t v = hist[c * 1024 + d]; hist[c * 1024 + d] = run; run += v; }
                pool.run(nc, [&](size_t c) {
                    uint32_t* h = hist.data() + c * 1024;
                    const size_t b = c * per, e = std::min(n, b + per);
                    for (size_t i = b; i < e; i++) { const uint32_t d = h[(code[i] >> shift) & 1023u]++; code2[d] = code[i]; idx2[d] = idx[i]; }
                });
                code.swap(code2); idx.swap(idx2);
            }
        }
        // Treelets: runs with equal top 12 bits (bvh.rs:240-265).  Each one is emitted into its own node array
        // (its slice of `order` starts at the treelet's first sorted position, as in the sequential build).
        struct Treelet { size_t start, count; std::vector<BuildNode> nodes; int root; };
        std::vector<Treelet> tl;
        for (size_t start = 0, end = 1; end <= n; end++) {
            if (end == n || ((code[start] ^ code[end]) & 0x3FFC0000u)) { tl.push_back({start, end - start, {}, -1}); start = end; }
        }
        pool.run(tl.size(), [&](size_t t) {
            Treelet& T = tl[t];
            uint32_t ordered = (uint32_t)T.start;
            T.nodes.reserve(2 * (T.count / std::max<size_t>(1, max_prims / 4)) + 8);
            T.root = emit(T.nodes, code.data() + T.start, idx.data() + T.start, T.count, boxes, max_prims, ordered, 17);
        });
        size_t total = 0;
        for (const Treelet& T : tl) total += T.nodes.size();
        nodes.clear(); nodes.reserve(total + 2 * tl.size() + 8);
        std::vector<int> treelets;
        for (Treelet& T : tl) {
            const int base = (int)nodes.size();
            for (BuildNode bn : T.nodes) { if (bn.left >= 0) { bn.left += base; bn.right += base; } nodes.push_back(bn); }
            treelets.push_back(T.root + base);
        }
        total_nodes = nodes.size();
        root = upper_sah(treelets.data(), treelets.size(), 0);
        total_nodes = nodes.size();
    }

    // emit_lbvh, bvh.rs:278-347
    int emit(std::vector<BuildNode>& nodes, const uint32_t* code, const uint32_t* idx, size_t n, const raw_vector<Box>& boxes, size_t max_prims, uint32_t& ordered, int bit) {
        while (true) {
            if (bit == -1 || n < max_prims) {
                BuildNode bn; bn.box = Box::none(); bn.first = ordered; bn.count = (uint32_t)n;
                for (size_t i = 0; i < n; i++) { order[ordered + i] = idx[i]; bn.box.grow(boxes[idx[i]]); }
                ordered += (uint32_t)n;
                nodes.push_back(bn);
                return (int)nodes.size() - 1;
            }
            const uint32_t mask = 1u << bit;
            if ((code[0] & mask) == (code[n - 1] & mask)) { bit--; continue; }
            size_t s = 0, e = n - 1;
            while (s + 1 != e) { size_t mid = (s + e) / 2; if ((code[s] & mask) == (code[mid] & mask)) s = mid; else e = mid; }
            const int me = (int)nodes.size();
            nodes.push_back(BuildNode());
            int l = emit(nodes, code, idx, e, boxes, max_prims, ordered, bit - 1);
            int r = emit(nodes, code + e, idx + e, n - e, boxes, max_prims, ordered, bit - 1);
            BuildNode& bn = nodes[me];
            bn.left = l; bn.right = r; bn.axis = (uint8_t)(bit % 3);
            bn.box = nodes[l].box; bn.box.grow(nodes[r].box);
            return me;
        }
    }

    // build_upper_sah, bvh.rs:350-427
    int upper_sah(int* roots, size_t n, int depth) {
        if (n == 1) return roots[0];
        const int me = (int)nodes.size();
        nodes.push_back(BuildNode());
        Box bounds = Box::none(), cb = Box::none();
        for (size_t i = 0; i < n; i++) {
            const Box& b = nodes[roots[i]].box;
            bounds.grow(b);
            double c[3]; for (int k = 0; k < 3; k++) c[k] = 0.5 * (b.mn[k] + b.mx[k]);
            cb.grow_pt(c);
        }
        const double dx = cb.mx[0] - cb.mn[0], dy = cb.mx[1] - cb.mn[1], dz = cb.mx[2] - cb.mn[2];
        const int dim = (dx > dy && dz > dz) ? 0 : (dy > dz ? 1 : 2);                  // bounds.rs:125-130 (sic)
        auto bucket = [&](int r) -> size_t {
            const Box& b = nodes[r].box;
            double c = (b.mn[dim] + b.mx[dim]) * 0.5;
            double b0 = (c - cb.mn[dim]) / (cb.mx[dim] - cb.mn[dim]);
            size_t k = (size_t)sat_u32(12.0 * b0);
            return k == 12 ? 11 : k;
        };
        size_t cnt[12] = {0}; Box bb[12]; for (auto& b : bb) b = Box::none();
        for (size_t i = 0; i < n; i++) {
            size_t k = bucket(roots[i]);
            if (k > 11) throw Error(LGB_ERR_INVALID, "SAH bucket index out of range (the reference would panic)");
            cnt[k]++; bb[k].grow(nodes[roots[i]].box);
        }
        double cost[12];
        for (int i = 0; i < 12; i++) {
            Box b0 = Box::none(), b1 = Box::none(); size_t c0 = 0, c1 = 0;
            for (int j = 0; j <= i; j++) { b0.grow(bb[j]); c0 += cnt[j]; }
            for (int j = i + 1; j < 12; j++) { b1.grow(bb[j]); c1 += cnt[j]; }
            cost[i] = 0.125 + ((double)c0 * b0.area() + (double)c1 * b1.area()) / bounds.area();
        }
        int best = 0;
        for (int i = 0; i < 12; i++) if (cost[i] < cost[best]) best = i;
        int* mid = std::partition(roots, roots + n, [&](int r) { return bucket(r) <= (size_t)best; });
        const size_t nlo = (size_t)(mid - roots);
        if (nlo == 0 || nlo == n)
            throw Error(LGB_ERR_INVALID, "degenerate SAH split: treelet centroids coincide in y and z; the reference does not terminate (bvh.rs:376-424)");
        int l = upper_sah(roots, nlo, depth + 1);
        int r = upper_sah(mid, n - nlo, depth + 1);
        BuildNode& bn = nodes[me];
        bn.left = l; bn.right = r; bn.axis = (uint8_t)dim;
        bn.box = nodes[l].box; bn.box.grow(nodes[r].box);
        return me;
    }
};

// Transform3::transform_bounds, transform.rs:219-240 (m is cgmath column-major: column c at m[4c .. 4c+3]).
inline double bmin(double a, double b) { return a < b ? a : b; }     // transform.rs:308-309
inline double bmax(double a, double b) { return a < b ? b : a; }
inline Box transform_bounds(const double m[16], const Box& b) {
    Box o;
    for (int r = 0; r < 3; r++) {
        const double xa = m[0 + r] * b.mn[0], xb = m[0 + r] * b.mx[0];
        const double ya = m[4 + r] * b.mn[1], yb = m[4 + r] * b.mx[1];
        const double za = m[8 + r] * b.mn[2], zb = m[8 + r] * b.mx[2];
        const double lo = bmin(xa, xb) + bmin(ya, yb) + bmin(za, zb) + m[12 + r];
        const double hi = bmax(xa, xb) + bmax(ya, yb) + bmax(za, zb) + m[12 + r];
        o.mn[r] = lo < hi ? lo : hi; o.mx[r] = lo < hi ? hi : lo;          // Bounds3::new, bounds.rs:37-42
    }
    return o;
}

// A level being assembled: its reference tree plus what each primitive is.
struct Level {
    LevelTree tree;
    raw_vector<Box> boxes;
    raw_vector<uint32_t> refs;                // prim ref per primitive (instances: index into `children`)
    std::vector<std::unique_ptr<Level>> children;
    std::vector<uint32_t> child_instance;     // instance slot per child
    size_t per_node = 0;                      // max_prims_per_node argument of BVHAccel::new for this level (bvh.rs:141-162)
    // The level's root box: the union of its primitive bounds (bvh.rs:212-213); min / max folds do not depend on the tree.
    Box bounds() const {
        lgb::Pool& pool = lgb::Pool::get();
        const size_t n = boxes.size(), nc = std::max<size_t>(1, pool.chunks_of(n, 1 << 14));
        std::vector<Box> part(nc, Box::none());
        pool.for_range(n, 1 << 14, [&](size_t b, size_t e, size_t c) { for (size_t i = b; i < e; i++) part[c].grow(boxes[i]); });
        Box all = Box::none();
        for (const Box& b : part) all.grow(b);
        return all;
    }
    void build_trees() {                      // nested levels first, as the reference's recursion does
        for (auto& c : children) c->build_trees();
        tree.build(boxes, per_node);
    }
};

using HostLevel = Level;                   // FlatScene has a nested type of the same name

inline float f32_down(double v) { float f = (float)v; if ((double)f > v) f = std::nextafterf(f, -INFINITY); return f; }
inline float f32_up(double v) { float f = (float)v; if ((double)f < v) f = std::nextafterf(f, INFINITY); return f; }

struct Flattener {
    const Scene& scene;
    const BuildOptions& opt;
    FlatScene& out;
    std::vector<int> mat_cache_kind;
    uint32_t next_id = 0;

    uint32_t material_index(const Material& m) {
        if (m.kind < Material::Matte || m.kind > Material::Mirror) throw Error(LGB_ERR_INVALID, "unknown material kind");
        for (size_t i = 0; i < out.materials.size(); i++) {
            const lgb_material& q = out.materials[i];
            if ((int)q.kind == m.kind && q.roughness == m.roughness && q.roughness_v == m.roughness_v && !std::memcmp(q.kd, m.kd, 24) && !std::memcmp(q.ks, m.ks, 24)) return (uint32_t)i;
        }
        lgb_material q{}; std::memcpy(q.kd, m.kd, 24); std::memcpy(q.ks, m.ks, 24); q.roughness = m.roughness; q.roughness_v = m.roughness_v; q.kind = (uint32_t)m.kind;
        out.materials.push_back(q);
        return (uint32_t)out.materials.size() - 1;
    }

    // BVHAccel::from_mesh, bvh.rs:141-148
    std::unique_ptr<Level> level_from_mesh(size_t mesh_index, bool has_mat, const Material& mat) {
        if (mesh_index >= scene.meshes.size()) throw Error(LGB_ERR_INVALID, "mesh reference out of range (Scene::obj(...).unwrap() would panic)");
        const ObjData& m = scene.meshes[mesh_index];
        const size_t ntri = m.faces.size() / 3;
        const bool has_n = !m.normals.empty();
        const uint32_t mi = material_index(has_mat ? mat : Material::default_());   // bvh.rs:513-515, material/mod.rs:15-17
        auto lv = std::make_unique<Level>();
        lv->boxes.resize(ntri); lv->refs.resize(ntri);
        const size_t base = out.triangles.size();
        out.triangles.resize(base + ntri); out.triangle_material.resize(base + ntri); out.triangle_id.resize(base + ntri);
        const bool track_n = has_n || !out.tri_normals.empty();
        if (track_n) {
            const size_t had = out.tri_has_normals.size();
            out.tri_normals.resize(base + ntri); out.tri_has_normals.resize(base + ntri);
            std::fill(out.tri_has_normals.begin() + had, out.tri_has_normals.begin() + base, (uint8_t)0);   // earlier meshes without normals
        }
        const uint32_t id0 = next_id; next_id += (uint32_t)ntri;
        std::atomic<bool> bad_index{false};
        lgb::Pool::get().for_range(ntri, 1 << 14, [&](size_t t0, size_t t1, size_t) {
          for (size_t t = t0; t < t1; t++) {
            if ((size_t)m.faces[3 * t] * 3 + 2 >= m.positions.size() || (size_t)m.faces[3 * t + 1] * 3 + 2 >= m.positions.size() ||
                (size_t)m.faces[3 * t + 2] * 3 + 2 >= m.positions.size()) { bad_index.store(true); continue; }
            lgb_triangle& tr = out.triangles[base + t];
            const float* p0 = &m.positions[3 * (size_t)m.faces[3 * t]], *p1 = &m.positions[3 * (size_t)m.faces[3 * t + 1]], *p2 = &m.positions[3 * (size_t)m.faces[3 * t + 2]];
            Box b;
            for (int k = 0; k < 3; k++) {
                tr.p0[k] = p0[k]; tr.p1[k] = p1[k]; tr.p2[k] = p2[k];
                double a = p0[k], c = p1[k], e = p2[k];                 // triangle.rs:157-159
                double lo = a < c ? a : c, hi = a < c ? c : a;
                b.mn[k] = lo < e ? lo : e; b.mx[k] = hi < e ? e : hi;
            }
            if (has_n) {
                if ((size_t)m.normal_faces[3 * t] * 3 + 2 >= m.normals.size() || (size_t)m.normal_faces[3 * t + 1] * 3 + 2 >= m.normals.size() ||
                    (size_t)m.normal_faces[3 * t + 2] * 3 + 2 >= m.normals.size()) { bad_index.store(true); continue; }
                lgb_tri_normals& q = out.tri_normals[base + t];
                for (int k = 0; k < 3; k++) {
                    q.n0[k] = m.normals[3 * (size_t)m.normal_faces[3 * t] + k];
                    q.n1[k] = m.normals[3 * (size_t)m.normal_faces[3 * t + 1] + k];
                    q.n2[k] = m.normals[3 * (size_t)m.normal_faces[3 * t + 2] + k];
                }
                out.tri_has_normals[base + t] = 1;
            } else if (track_n) out.tri_has_normals[base + t] = 0;
            out.triangle_material[base + t] = mi;
            out.triangle_id[base + t] = id0 + (uint32_t)t;
            lv->boxes[t] = b;
            lv->refs[t] = LGB_PRIM_REF(LGB_PRIM_TRIANGLE, base + t);
          }
        });
        if (bad_index.load()) throw Error(LGB_ERR_INVALID, "mesh face references a vertex or normal out of range");
        lv->per_node = ntri;
        return lv;
    }

    // BVHAccel::from_aggregate, bvh.rs:150-162
    std::unique_ptr<Level> level_from_aggregate(const Aggregate& ag, bool is_root) {
        (void)is_root;
        auto lv = std::make_unique<Level>();
        // Pass 1: canonical ids (SURVEY 8b: construction order, nested levels included) and array slots.  The nodes are 150-byte
        // records, so even reading their kinds is a 150 MB sweep for a million spheres: the chunks count their spheres / cuboids and
        // note their mesh / group nodes in parallel (1a), a short sequential walk over the chunks hands out the bases and builds the
        // nested levels in order (1b), and the chunks write ids and slots in parallel (1c).
        const size_t nn = ag.contents.size();
        lv->boxes.resize(nn); lv->refs.resize(nn);
        constexpr size_t kGrain = 1 << 13;
        const size_t n_chunks = lgb::Pool::get().chunks_of(nn, kGrain);                    // the partition for_range makes of [0, nn)
        const size_t per_chunk = n_chunks ? (nn + n_chunks - 1) / n_chunks : 0;
        struct ChunkInfo { uint32_t n_s = 0, n_c = 0; std::vector<uint32_t> nested; uint32_t id_base = 0, s_ord = 0, c_ord = 0; std::vector<uint32_t> nested_ids; };
        std::vector<ChunkInfo> chunks(n_chunks);
        lgb::Pool::get().for_range(nn, kGrain, [&](size_t b0, size_t e0, size_t c) {
            ChunkInfo& ci = chunks[c];
            for (size_t i = b0; i < e0; i++) {
                const Aggregate::Node::Kind k = ag.contents[i].kind;
                if (k == Aggregate::Node::Sphere) ci.n_s++;
                else if (k == Aggregate::Node::Cube || k == Aggregate::Node::Cuboid) ci.n_c++;
                else ci.nested.push_back((uint32_t)i);
            }
        });
        size_t n_s = 0, n_c = 0;       // ordinals among this level's own spheres / cuboids
        for (size_t c = 0; c < n_chunks; c++) {
            ChunkInfo& ci = chunks[c];
            ci.id_base = next_id; ci.s_ord = (uint32_t)n_s; ci.c_ord = (uint32_t)n_c;
            n_s += ci.n_s; n_c += ci.n_c;
            // ids inside the chunk: primitives before a nested node come first, then the nested level's own primitives
            size_t prev = c * per_chunk;
            for (uint32_t at : ci.nested) {
                const Aggregate::Node& n = ag.contents[at];
                next_id += (uint32_t)(at - prev);                  // the own primitives in [prev, at)
                ci.nested_ids.push_back(next_id);                  // id the next own primitive after `at` would have had before the nested level took its ids
                std::unique_ptr<Level> child = n.kind == Aggregate::Node::Mesh ? level_from_mesh(n.ref, n.has_mat, n.mat)
                                                                                : level_from_aggregate(ag.groups[n.ref], false);
                lgb_instance inst{};
                inst.identity = 1;
                for (int k = 0; k < 16; k++) inst.m[k] = inst.minv[k] = (k % 5 == 0) ? 1.0 : 0.0;
                const Box cb = child->bounds();
                if (n.kind == Aggregate::Node::Group) {
                    const Aggregate& g = ag.groups[n.ref];
                    inst.identity = g.transform.identity ? 1u : 0u;
                    inst.swap_backface = g.swap_backface_flag ? 1u : 0u;
                    std::memcpy(inst.m, g.transform.m, sizeof inst.m); std::memcpy(inst.minv, g.transform.minv, sizeof inst.minv);
                }
                lv->boxes[at] = transform_bounds(inst.m, cb);                  // BVHAccel::bound, bvh.rs:457-459
                out.instances.push_back(inst);
                lv->refs[at] = LGB_PRIM_REF(LGB_PRIM_INSTANCE, out.instances.size() - 1);
                lv->child_instance.push_back((uint32_t)out.instances.size() - 1);
                lv->children.push_back(std::move(child));
                ci.nested_ids.back() = next_id;                    // first id after the nested level
                prev = at + 1;
            }
            const size_t end = std::min(nn, (c + 1) * per_chunk);
            next_id += (uint32_t)(end - prev);
        }
        const size_t s_base = out.spheres.size(), c_base = out.cuboids.size();      // after the nested levels took theirs
        // (1c, the ids and slots of the chunk's own primitives, is a running count along the chunk: pass 2 below walks the same chunks
        // and keeps it in registers -- a third sweep over the 150-byte nodes and two arrays of a word per node are not needed)
        out.spheres.resize(s_base + n_s); out.sphere_material.resize(s_base + n_s); out.sphere_id.resize(s_base + n_s);
        out.cuboids.resize(c_base + n_c); out.cuboid_material.resize(c_base + n_c); out.cuboid_id.resize(c_base + n_c);
        // Pass 2 (all threads): primitive records and bounds.  Materials are interned through a small per-chunk
        // cache; a miss takes the lock.
        std::mutex mat_mutex;
        std::atomic<bool> failed{false};
        std::string fail_msg; int fail_status = LGB_ERR_INVALID;
        lgb::Pool::get().for_range(nn, kGrain, [&](size_t b0, size_t e0, size_t chunk) {
            const ChunkInfo& ci = chunks[chunk];
            uint32_t id = ci.id_base, so = ci.s_ord + (uint32_t)s_base, co = ci.c_ord + (uint32_t)c_base;
            size_t ni = 0;
            struct Cached { Material m; uint32_t index; };
            std::vector<Cached> cache;
            auto intern = [&](const Material& m) -> uint32_t {
                for (const Cached& c : cache)
                    if (c.m.kind == m.kind && c.m.roughness == m.roughness && c.m.roughness_v == m.roughness_v && !std::memcmp(c.m.kd, m.kd, 24) && !std::memcmp(c.m.ks, m.ks, 24)) return c.index;
                std::lock_guard<std::mutex> lock(mat_mutex);
                const uint32_t idx = material_index(m);
                if (cache.size() < 64) cache.push_back({m, idx});
                return idx;
            };
            try {
                for (size_t i = b0; i < e0; i++) {
                    const Aggregate::Node& n = ag.contents[i];
                    Box b;
                    if (n.kind == Aggregate::Node::Sphere) {
                        lgb_sphere s; for (int k = 0; k < 3; k++) { s.center[k] = n.a[k]; double lo = n.a[k] - n.r, hi = n.a[k] + n.r; b.mn[k] = lo < hi ? lo : hi; b.mx[k] = lo < hi ? hi : lo; }   // sphere.rs:73-77
                        s.radius = n.r;
                        const uint32_t at = so++;
                        out.spheres[at] = s; out.sphere_material[at] = intern(n.mat); out.sphere_id[at] = id++;
                        lv->refs[i] = LGB_PRIM_REF(LGB_PRIM_SPHERE, at);
                    } else if (n.kind == Aggregate::Node::Cube || n.kind == Aggregate::Node::Cuboid) {
                        lgb_cuboid c;
                        for (int k = 0; k < 3; k++) {
                            double p0 = n.a[k], p1 = n.kind == Aggregate::Node::Cube ? n.a[k] + n.r : n.b[k];   // cuboid.rs:18-30
                            c.min[k] = p0 < p1 ? p0 : p1; c.max[k] = p0 < p1 ? p1 : p0;                          // Bounds::new, bounds.rs:37-42
                            b.mn[k] = c.min[k]; b.mx[k] = c.max[k];
                        }
                        const uint32_t at = co++;
                        out.cuboids[at] = c; out.cuboid_material[at] = intern(n.mat); out.cuboid_id[at] = id++;
                        lv->refs[i] = LGB_PRIM_REF(LGB_PRIM_CUBOID, at);
                    } else { id = ci.nested_ids[ni++]; continue; }            // the nested level's primitives took the ids in between
                    lv->boxes[i] = b;
                }
            } catch (const Error& e) {
                std::lock_guard<std::mutex> lock(mat_mutex);
                if (!failed.exchange(true)) { fail_msg = e.what(); fail_status = e.status; }
            }
        });
        if (failed.load()) throw Error(fail_status, fail_msg);
        if (lv->boxes.empty()) throw Error(LGB_ERR_INVALID, "empty aggregate: the reference's BVH build does not terminate (bvh.rs:240,355-356)");
        lv->per_node = lv->boxes.size();
        return lv;
    }

};

// Emission of the built reference trees in pre-order (flatten_bvh_tree, bvh.rs:430-453).
struct Emitter {
    FlatScene& out;
    bool keep_levels;
    // ---- emission: reference tree in pre-order (flatten_bvh_tree, bvh.rs:430-453)
    static lgb_node node_box(const Box& b) {
        lgb_node n;
        for (int k = 0; k < 3; k++) { n.lo[k] = f32_down(b.mn[k]); n.hi[k] = f32_up(b.mx[k]); }
        n.a = 0; n.b = 0;
        return n;
    }
    void emit_node(const Level& lv, int bi) {
        const BuildNode& bn = lv.tree.nodes[bi];
        if (bn.left < 0) {
            lgb_node n = node_box(bn.box);
            n.a = (uint32_t)out.prim_refs.size(); n.b = LGB_LEAF_FLAG | bn.count;
            out.nodes.push_back(n);
            for (uint32_t i = 0; i < bn.count; i++) out.prim_refs.push_back(lv.refs[lv.tree.order[bn.first + i]]);    // bvh.rs:484
            return;
        }
        const uint32_t me = (uint32_t)out.nodes.size();
        out.nodes.push_back(node_box(bn.box));
        emit_node(lv, bn.left);
        const uint32_t second = (uint32_t)out.nodes.size();
        emit_node(lv, bn.right);
        out.nodes[me].a = second; out.nodes[me].b = bn.axis;
    }
    void dump_level(const Level& lv, uint32_t node_offset) {
        FlatScene::Level L; L.node_offset = node_offset;
        // pre-order walk of the reference tree with the reference's own leaf offsets
        // iterative pre-order producing (bounds, leaf, a, b)
        std::vector<int> stack{lv.tree.root};
        std::vector<size_t> fix;                        // interior slots waiting for their second child
        std::vector<int> fix_right;
        while (!stack.empty()) {
            int bi = stack.back(); stack.pop_back();
            const BuildNode& bn = lv.tree.nodes[bi];
            size_t slot = L.meta.size() / 3;
            while (!fix.empty() && fix_right.back() == bi) { L.meta[3 * fix.back() + 1] = (uint32_t)slot; fix.pop_back(); fix_right.pop_back(); }
            for (int k = 0; k < 3; k++) L.bounds.push_back(bn.box.mn[k]);
            for (int k = 0; k < 3; k++) L.bounds.push_back(bn.box.mx[k]);
            if (bn.left < 0) { L.meta.push_back(1); L.meta.push_back(bn.first); L.meta.push_back(bn.count & 0xFFFFu); }
            else {
                L.meta.push_back(0); L.meta.push_back(0); L.meta.push_back(bn.axis);
                fix.push_back(slot); fix_right.push_back(bn.right);
                stack.push_back(bn.right); stack.push_back(bn.left);
            }
        }
        L.order.assign(lv.tree.order.begin(), lv.tree.order.end());
        out.levels.push_back(std::move(L));
    }
    void emit_level(const Level& lv) {
        const uint32_t offset = (uint32_t)out.nodes.size();
        if (keep_levels) dump_level(lv, offset);
        emit_node(lv, lv.tree.root);
        for (size_t c = 0; c < lv.children.size(); c++) {
            out.instances[lv.child_instance[c]].root_node = (uint32_t)out.nodes.size();
            emit_level(*lv.children[c]);
        }
    }
};

}  // namespace

// lasgun::Camera -> lgb_camera: what lgb_scene_desc.camera and lgb_scene_set_camera take
static lgb_camera to_lgb_camera(const Camera& c) {
    lgb_camera o{};
    std::memcpy(o.origin, c.origin, 24); std::memcpy(o.view, c.view, 24);
    std::memcpy(o.up, c.up, 24); std::memcpy(o.aux, c.aux, 24);
    o.image_plane_height = c.image_plane_height; o.pixel_separation = c.pixel_separation;
    o.sample_distance = c.distance; o.supersampling_root = (uint32_t)c.root;
    return o;
}

FlatScene flatten(const Scene& scene, const BuildOptions& opt) {
    auto t0 = std::chrono::steady_clock::now();
    FlatScene out;
    Flattener f{scene, opt, out, {}, 0};
    std::unique_ptr<Level> root = f.level_from_aggregate(scene.root, true);
    out.root = lgb_instance{};
    out.root.identity = scene.root.transform.identity ? 1u : 0u;
    out.root.swap_backface = scene.root.swap_backface_flag ? 1u : 0u;
    std::memcpy(out.root.m, scene.root.transform.m, sizeof out.root.m); std::memcpy(out.root.minv, scene.root.transform.minv, sizeof out.root.minv);
    const double t_levels = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    {
        const Box wb = root->bounds();                       // = the reference root box, in the root aggregate's coordinates
        for (int k = 0; k < 3; k++) { out.bounds_lo[k] = wb.mn[k]; out.bounds_hi[k] = wb.mx[k]; }
    }
    out.keep_levels = opt.keep_levels;
    out.pending = std::shared_ptr<void>(root.release(), [](void* p) { delete static_cast<Level*>(p); });
    bool transformed = !out.root.identity || out.root.swap_backface;
    for (const lgb_instance& in : out.instances) transformed |= !in.identity || in.swap_backface;
    if (!opt.lazy_tree || transformed) out.build_reference_tree();      // nested spaces are derived from the tree: no lazy mode for them
    if (std::getenv("LGB_TIMING")) std::fprintf(stderr, "[flatten] primitives and levels %.1f ms, reference trees %s %.1f ms\n", t_levels, out.tree_built ? "built" : "deferred",
                                                 std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count() - t_levels);
    out.prim_count = f.next_id;
    out.flags = 0;
    if (scene.lights.size() > LGB_MAX_LIGHTS) throw Error(LGB_ERR_UNSUPPORTED, "more than LGB_MAX_LIGHTS point lights");
    for (const Scene::Light& l : scene.lights) {
        lgb_light q; std::memcpy(q.position, l.position, 24); std::memcpy(q.intensity, l.intensity, 24); std::memcpy(q.falloff, l.falloff, 24);
        out.lights.push_back(q);
    }
    out.camera = to_lgb_camera(scene.camera);
    std::memcpy(out.ambient, scene.ambient, 24); std::memcpy(out.bg_inner, scene.bg_inner, 24); std::memcpy(out.bg_outer, scene.bg_outer, 24);
    out.bg_scale = scene.bg_scale; out.recursion = scene.recursion;
    out.build_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    return out;
}

// BVHAccel::from for every level (bvh.rs:135-453) and the pre-order emission.  Lazy scenes reach this only through the
// reference_tree callback, i.e. when the device met an exact-t tie.
void FlatScene::build_reference_tree() {
    if (tree_built) return;
    HostLevel* root = static_cast<HostLevel*>(pending.get());
    if (!root) throw Error(LGB_ERR_INVALID, "FlatScene: no pending levels");
    root->build_trees();
    Emitter em{*this, keep_levels};
    em.emit_level(*root);
    tree_built = true;
    pending.reset();
}
static int reference_tree_trampoline(void* user, lgb_reference_tree* out) {
    FlatScene* f = static_cast<FlatScene*>(user);
    try { f->build_reference_tree(); } catch (...) { return -1; }
    out->nodes = f->nodes.data(); out->n_nodes = f->nodes.size();
    out->prim_refs = f->prim_refs.data(); out->n_prim_refs = f->prim_refs.size();
    out->instances = f->instances.data(); out->n_instances = f->instances.size();
    return 0;
}

void FlatScene::describe(lgb_scene_desc* d) const {
    std::memset(d, 0, sizeof *d);
    d->abi_version = LGB_ABI_VERSION; d->flags = flags;
    if (tree_built) {
        d->nodes = nodes.data(); d->n_nodes = nodes.size();
        d->prim_refs = prim_refs.data(); d->n_prim_refs = prim_refs.size();
    } else {                                                  // lazy: the device asks for the tree if it ever needs it
        d->reference_tree = reference_tree_trampoline; d->reference_tree_user = const_cast<FlatScene*>(this);
    }
    std::memcpy(d->bounds_lo, bounds_lo, 24); std::memcpy(d->bounds_hi, bounds_hi, 24);
    d->spheres = spheres.data(); d->n_spheres = spheres.size(); d->sphere_material = sphere_material.data(); d->sphere_id = sphere_id.data();
    d->cuboids = cuboids.data(); d->n_cuboids = cuboids.size(); d->cuboid_material = cuboid_material.data(); d->cuboid_id = cuboid_id.data();
    d->triangles = triangles.data(); d->n_triangles = triangles.size(); d->triangle_material = triangle_material.data(); d->triangle_id = triangle_id.data();
    d->tri_normals = tri_normals.empty() ? nullptr : tri_normals.data();
    d->tri_has_normals = tri_has_normals.empty() ? nullptr : tri_has_normals.data();
    if (tree_built) { d->instances = instances.data(); d->n_instances = instances.size(); }
    d->root = root;
    d->materials = materials.data(); d->n_materials = materials.size();
    d->lights = lights.data(); d->n_lights = lights.size();
    d->camera = camera;
    std::memcpy(d->ambient, ambient, 24); std::memcpy(d->bg_inner, bg_inner, 24); std::memcpy(d->bg_outer, bg_outer, 24);
    d->bg_scale = bg_scale; d->recursion = recursion;
}

// ------------------------------------------------------------------ Accel / capture
static std::mutex g_ctx_mutex;
static lgb_ctx* g_ctx = nullptr;
lgb_ctx* default_context() {
    std::lock_guard<std::mutex> lock(g_ctx_mutex);
    if (!g_ctx) {
        // LASGUN_DEVICES: "all" = every visible GPU as one device group (the reference takes every core, lib.rs:165), a comma
        // separated list = those, unset = device 0 alone (a process launched once per GPU must not grab its neighbours')
        std::vector<int> devs;
        if (const char* e = std::getenv("LASGUN_DEVICES")) {
            if (std::string(e) == "all") { for (int i = 0; i < lgb_device_count(); i++) devs.push_back(i); }
            else for (const char* q = e; *q;) { char* end = nullptr; const long v = std::strtol(q, &end, 10); if (end == q) break; devs.push_back((int)v); q = *end ? end + 1 : end; }
        }
        int rc = devs.size() > 1 ? lgb_init_devices((int)devs.size(), devs.data(), &g_ctx) : lgb_init(devs.empty() ? 0 : devs[0], &g_ctx);
        if (rc) throw Error(rc, std::string("lasgun: cannot open the GPU: ") + lgb_last_error(nullptr));
    }
    return g_ctx;
}

std::unique_ptr<Accel> Accel::from(const Scene& scene, lgb_ctx* ctx, const BuildOptions& opt) {
    auto a = std::make_unique<Accel>();
    a->ctx = ctx ? ctx : default_context();
    a->flat = flatten(scene, opt);
    lgb_scene_desc d; a->flat.describe(&d);
    d.expected_film_pixels = opt.expected_film_pixels;
    int rc = lgb_scene_create(a->ctx, &d, &a->dev);
    if (rc) throw Error(rc, std::string("lgb_scene_create: ") + lgb_last_error(a->ctx));
    return a;
}
Accel::~Accel() { if (dev) lgb_scene_destroy(dev); }

void capture(const Scene& scene, Film& film) {                   // lib.rs:55-104
    BuildOptions opt; opt.lazy_tree = true;                      // the reference BVH is built only if a ray meets an exact-t tie
    opt.expected_film_pixels = (uint64_t)film.w * film.h < (1ull << 32) ? film.w * film.h : 0u;      // capture knows its film: lets the device skip a BVH no ray will walk
    std::unique_ptr<Accel> root = Accel::from(scene, nullptr, opt);
    int rc = lgb_capture(root->ctx, root->dev, film.w, film.h, film.data(), nullptr);
    if (rc) throw Error(rc, std::string("lgb_capture: ") + lgb_last_error(root->ctx));
}
void capture_subset(size_t k, size_t n, const Accel& root, Film& film) {   // lib.rs:110-162
    int rc = lgb_capture_subset(root.ctx, root.dev, (uint32_t)k, (uint32_t)n, film.w, film.h, film.data(), nullptr);
    if (rc) throw Error(rc, std::string("lgb_capture_subset: ") + lgb_last_error(root.ctx));
}
Film render(const Scene& scene, uint32_t width, uint32_t height) {          // lib.rs:46-50
    Film film(width, height);
    capture(scene, film);
    return film;
}

}  // namespace lasgun

// ==================================================================== flat C wrappers (ctypes)
using namespace lasgun;
namespace {
struct HostScene {
    Scene scene;
    std::vector<std::unique_ptr<Aggregate>> pending;   // handle 0 is scene.root
    std::string error;
    Aggregate& agg(int h) { return h == 0 ? scene.root : *pending[(size_t)h - 1]; }
};
thread_local std::string g_host_error;
Material mk(int kind, const double* kd, const double* ks, double rough, double rough_v) {
    Material m; m.kind = kind; std::memcpy(m.kd, kd, 24); std::memcpy(m.ks, ks, 24); m.roughness = rough; m.roughness_v = rough_v; return m;
}
template <class F> int guarded(F&& f) {
    try { f(); return LGB_OK; }
    catch (const Error& e) { g_host_error = e.what(); return e.status; }
    catch (const std::exception& e) { g_host_error = e.what(); return LGB_ERR_INVALID; }
}
}  // namespace

extern "C" {
const char* lgh_last_error() { return g_host_error.c_str(); }
void* lgh_scene_new() { return new HostScene(); }
void lgh_scene_free(void* s) { delete (HostScene*)s; }
void lgh_set_perspective_camera(void* s, double fov) { ((HostScene*)s)->scene.set_perspective_camera(fov); }
void lgh_set_orthographic_camera(void* s, double h) { ((HostScene*)s)->scene.set_orthographic_camera(h); }
void lgh_look_at(void* s, const double* o, const double* l, const double* u) { ((HostScene*)s)->scene.camera.look_at(o, l, u); }
int lgh_set_supersampling(void* s, int base) { return guarded([&] { ((HostScene*)s)->scene.camera.set_supersampling((uint8_t)base); }); }
// The lgb_camera of a camera set up as a scene's: the perspective or orthographic constructor, look_at if origin, look and up are
// given, then set_supersampling -- the reference's arithmetic, so a camera moved to later equals a scene built with it, bit for bit.
int lgh_camera_describe(int perspective, double param, const double* origin, const double* look, const double* up, int supersampling, lgb_camera* out) {
    return guarded([&] {
        Camera c = perspective ? Camera::perspective(param) : Camera::orthographic(param);
        if (origin && look && up) c.look_at(origin, look, up);
        c.set_supersampling((uint8_t)supersampling);
        *out = to_lgb_camera(c);
    });
}
void lgh_set_ambient_light(void* s, const double* c) { ((HostScene*)s)->scene.set_ambient_light(c); }
void lgh_set_radial_background(void* s, const double* in, const double* out, double scale) { ((HostScene*)s)->scene.set_radial_background(in, out, scale); }
void lgh_set_max_recursion_depth(void* s, uint32_t depth) { ((HostScene*)s)->scene.set_max_recursion_depth(depth); }
void lgh_set_mesh_smoothing(void* s, int on) { ((HostScene*)s)->scene.set_mesh_smoothing(on != 0); }
void lgh_add_point_light(void* s, const double* p, const double* i, const double* f) { ((HostScene*)s)->scene.add_point_light(p, i, f); }
int lgh_add_mesh(void* s, const float* pos, uint64_t nv, const uint32_t* vi, uint64_t ntri, const float* nrm, uint64_t nn, const uint32_t* ni, int64_t* ref_out) {
    return guarded([&] {
        ObjData m; m.positions.assign(pos, pos + 3 * nv); m.faces.assign(vi, vi + 3 * ntri);
        if (nrm && nn) { m.normals.assign(nrm, nrm + 3 * nn); m.normal_faces.assign(ni, ni + 3 * ntri); }
        *ref_out = (int64_t)((HostScene*)s)->scene.add_obj(std::move(m)).index;
    });
}
int lgh_agg_new(void* s) { HostScene* h = (HostScene*)s; h->pending.emplace_back(new Aggregate()); return (int)h->pending.size(); }
void lgh_agg_add_sphere(void* s, int ag, const double* c, double r, int kind, const double* kd, const double* ks, double rough, double rough_v) {
    ((HostScene*)s)->agg(ag).add_sphere(c, r, mk(kind, kd, ks, rough, rough_v));
}
void lgh_agg_add_spheres(void* s, int ag, uint64_t n, const double* c, const double* r, int nmat, const int* kinds, const double* kd,
                         const double* ks, const double* rough, const double* rough_v, const int* mat_index) {
    Aggregate& a = ((HostScene*)s)->agg(ag); (void)nmat;
    a.contents.reserve(a.contents.size() + n);
    for (uint64_t i = 0; i < n; i++) { int m = mat_index[i]; a.add_sphere(c + 3 * i, r[i], mk(kinds[m], kd + 3 * m, ks + 3 * m, rough[m], rough_v[m])); }
}
void lgh_agg_add_cube(void* s, int ag, const double* o, double dim, int kind, const double* kd, const double* ks, double rough, double rough_v) {
    ((HostScene*)s)->agg(ag).add_cube(o, dim, mk(kind, kd, ks, rough, rough_v));
}
void lgh_agg_add_box(void* s, int ag, const double* a, const double* b, int kind, const double* kd, const double* ks, double rough, double rough_v) {
    ((HostScene*)s)->agg(ag).add_box(a, b, mk(kind, kd, ks, rough, rough_v));
}
void lgh_agg_add_mesh(void* s, int ag, int64_t mesh, int has_mat, int kind, const double* kd, const double* ks, double rough, double rough_v) {
    if (has_mat) ((HostScene*)s)->agg(ag).add_obj_of(ObjRef{(size_t)mesh}, mk(kind, kd, ks, rough, rough_v));
    else ((HostScene*)s)->agg(ag).add_obj(ObjRef{(size_t)mesh});
}
void lgh_agg_add_group(void* s, int parent, int child) {
    HostScene* h = (HostScene*)s;
    Aggregate moved = std::move(*h->pending[(size_t)child - 1]);
    h->agg(parent).add_group(std::move(moved));
}
void lgh_agg_swap_backface(void* s, int ag) { ((HostScene*)s)->agg(ag).swap_backface(); }
void lgh_agg_translate(void* s, int ag, const double* d) { ((HostScene*)s)->agg(ag).translate(d); }
void lgh_agg_scale(void* s, int ag, double x, double y, double z) { ((HostScene*)s)->agg(ag).scale(x, y, z); }
void lgh_agg_rotate_axis(void* s, int ag, int axis, double deg) {
    Aggregate& a = ((HostScene*)s)->agg(ag);
    if (axis == 0) a.rotate_x(deg); else if (axis == 1) a.rotate_y(deg); else a.rotate_z(deg);
}
void lgh_agg_rotate(void* s, int ag, double deg, const double* axis) { ((HostScene*)s)->agg(ag).rotate(deg, axis); }

// Accel::from minus the upload: build + flatten on the host.
void* lgh_flatten(void* s, int keep_levels, int lazy_tree) {
    FlatScene* out = nullptr;
    int rc = guarded([&] {
        BuildOptions o; o.keep_levels = keep_levels != 0; o.lazy_tree = lazy_tree != 0;
        out = new FlatScene(flatten(((HostScene*)s)->scene, o));
    });
    (void)rc;
    return out;
}
void lgh_flat_free(void* f) { delete (FlatScene*)f; }
int lgh_flat_tree_built(void* f) { return ((FlatScene*)f)->tree_built ? 1 : 0; }
int lgh_flat_build_tree(void* f) { return guarded([&] { ((FlatScene*)f)->build_reference_tree(); }); }
void lgh_flat_describe(void* f, lgb_scene_desc* out) { ((FlatScene*)f)->describe(out); }
double lgh_flat_build_ms(void* f) { return ((FlatScene*)f)->build_ms; }
uint32_t lgh_flat_prim_count(void* f) { return ((FlatScene*)f)->prim_count; }
uint64_t lgh_flat_level_count(void* f) { return ((FlatScene*)f)->levels.size(); }
int lgh_flat_level_dims(void* f, uint64_t level, uint64_t* n_nodes, uint64_t* n_prims, uint32_t* node_offset) {
    FlatScene* fs = (FlatScene*)f;
    if (level >= fs->levels.size()) return LGB_ERR_INVALID;
    *n_nodes = fs->levels[level].meta.size() / 3; *n_prims = fs->levels[level].order.size(); *node_offset = fs->levels[level].node_offset;
    return LGB_OK;
}
int lgh_flat_level_dump(void* f, uint64_t level, double* bounds, uint32_t* meta, uint64_t* order) {
    FlatScene* fs = (FlatScene*)f;
    if (level >= fs->levels.size()) return LGB_ERR_INVALID;
    const FlatScene::Level& L = fs->levels[level];
    std::memcpy(bounds, L.bounds.data(), L.bounds.size() * 8); std::memcpy(meta, L.meta.data(), L.meta.size() * 4); std::memcpy(order, L.order.data(), L.order.size() * 8);
    return LGB_OK;
}
// capture(scene, film) through the C++ mirror (lib.rs:55): build + flatten + upload + render + readback.
int lgh_capture(void* s, uint32_t w, uint32_t h, uint8_t* rgba) {
    return guarded([&] { Film film(w, h, rgba); capture(((HostScene*)s)->scene, film); });
}
}  // extern "C"
