// glass_oracle.cpp — the f64 ORACLE (oracle/rt_oracle.cpp) with the dielectric material (brdf 3, DESIGN §3e) added.
//
// TEST INFRASTRUCTURE ONLY.  The parity tests of the glass material (tests/test_dielectric_cpu.py,
// tests/test_gpu_dielectric.py) build it through tests/glass_oracle.py into a temporary directory.  Everything but the
// dielectric is oracle/rt_oracle.cpp as it stands, so it keeps that file's contract and its citations; oracle/ stays the
// pinned reference for every other test.  What the dielectric adds: B_DIELECTRIC in Scene::reflected_radiance (the same
// contract as k_shade), Hit::dir (the true direction, which a mirror in front does not hand down), and
// orient_dielectric (the loader's mesh orientation rule, restated independently).
//
// PARITY PINS: the reference (Rust) cannot be compiled here (no cargo/rustc) and holds no golden vectors; its
// only unit test (`test_octants`, src/geometry.rs:1115-1131) pins octant numbering and is reproduced in
// tests/test_oracle_pins.py.  What the reference DOES ship are three images its own renderer wrote
// (examples/cornell_box.png, examples/cubes.png, raytracer.gif); tests/test_reference_pins.py checks that this
// oracle, in the reference's real mode (octree traversal + live NEE), reproduces them region by region on the
// oracle-vs-oracle noise floor (50x50 tile means 0.26 % / 0.41 %, channel means 0.03 %, noise level 0.03 %,
// clamp loss and firefly count) — fixtures in tests/golden/reference_pins.npz, generator make_reference_pins.py.
// Still UNPINNED by any reference output: individual random sequences (the reference is OS-seeded), the dead
// "MIS" branch (no image of it exists), Phong and mesh lights (no reference scene uses them).
// The reference's RNG is rand 0.8.5 (Cargo.lock:556-557; ChaCha12 thread_rng, OS-seeded,
// source not under /root/reference).  Its sequences cannot be matched, only its
// distributions; this oracle draws from Philox4x32-10 (Salmon et al. 2011) with a
// documented (pixel, sample, depth, block) counter so that it and the CUDA path consume
// IDENTICAL random numbers (see DESIGN.md "RNG contract").
//
// Every function cites the reference file:line it restates.  Arithmetic is f64 in the
// reference's own expression order; build with -ffp-contract=off (rustc never contracts).
//
// Modes:
//   accel  0 = octree_faithful (Octree::intersect, src/geometry.rs:1237-1295, quirks kept)
//          1 = exact           (Mesh::intersect brute-force branch, src/geometry.rs:887-903,
//                               accelerated by an exact median-split BVH; same nearest hit)
//   estimator 0 = live NEE (src/scene.rs:217-229), 1 = dead "MIS" branch (src/scene.rs:189-216)

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <fstream>
#include <limits>
#include <map>
#include <sstream>
#include <string>
#include <thread>
#include <tuple>
#include <vector>

// ORACLE_F32 (liboracle_f32.so, `make liboracle_f32.so`): the SAME restatement with every stored quantity — scene data, rays,
// hit records, accumulators — in fp32, so that tests can ask "does the f64 answer survive fp32 rounding of the inputs?" for a
// ray on which the GPU (which stores fp32) and the f64 oracle disagree.  Only the intersection hooks (or_primary_rays /
// or_trace_rays) are meaningful in this build: the reference leaves a surface through a 1e-5 offset that fp32 cannot resolve at
// x ~ 100, so rendering with it self-intersects (the GPU handles that case analytically, intersect.cuh).  The C entry points then
// take float* where they take double* here; oracle.py (OracleScene(..., f32=True)) passes float32 arrays.
#ifdef ORACLE_F32
#define double float
#endif

namespace {

constexpr double PI = 3.14159265358979323846264338327950288;       // std::f64::consts::PI
constexpr double FRAC_1_PI = 0.318309886183790671537767526745028724;  // FRAC_1_PI

// ---------------------------------------------------------------- Vec3 (src/geometry.rs:21-134)
struct Vec3 {
    double x, y, z;
};
inline Vec3 V(double x, double y, double z) { return {x, y, z}; }
inline Vec3 operator-(const Vec3& a) { return {-a.x, -a.y, -a.z}; }
inline Vec3 operator+(const Vec3& a, const Vec3& b) { return {a.x + b.x, a.y + b.y, a.z + b.z}; }
inline Vec3 operator-(const Vec3& a, const Vec3& b) { return {a.x - b.x, a.y - b.y, a.z - b.z}; }
inline Vec3 operator*(const Vec3& a, double s) { return {a.x * s, a.y * s, a.z * s}; }
inline Vec3 operator*(double s, const Vec3& a) { return {s * a.x, s * a.y, s * a.z}; }
inline Vec3 operator/(const Vec3& a, double s) { return {a.x / s, a.y / s, a.z / s}; }
inline Vec3& operator+=(Vec3& a, const Vec3& b) {
    a.x += b.x; a.y += b.y; a.z += b.z;
    return a;
}
inline double dot(const Vec3& a, const Vec3& b) { return a.x * b.x + a.y * b.y + a.z * b.z; }  // :65
inline double mag(const Vec3& a) { return std::sqrt(a.x * a.x + a.y * a.y + a.z * a.z); }      // :57
inline Vec3 norm(const Vec3& a) { return a / mag(a); }                                          // :61
inline Vec3 cross(const Vec3& a, const Vec3& v) {                                               // :69
    return {a.y * v.z - a.z * v.y, a.z * v.x - a.x * v.z, a.x * v.y - a.y * v.x};
}
inline Vec3 mult(const Vec3& a, const Vec3& b) { return {a.x * b.x, a.y * b.y, a.z * b.z}; }    // :77
inline bool equal_within(const Vec3& a, const Vec3& v, double e) {                               // :85
    return std::fabs(a.x - v.x) < e && std::fabs(a.y - v.y) < e && std::fabs(a.z - v.z) < e;
}
inline Vec3 flip_across(const Vec3& s, const Vec3& axis) { return 2.0 * dot(s, axis) * axis - s; }  // :99
inline double clampd(double x, double lo, double hi) { return x < lo ? lo : (x > hi ? hi : x); }  // :11
inline Vec3 clampv(const Vec3& a, double lo, double hi) {                                        // :103
    return {clampd(a.x, lo, hi), clampd(a.y, lo, hi), clampd(a.z, lo, hi)};
}
inline Vec3 rot_x(const Vec3& s, double a) {  // :111
    return {s.x, s.y * std::cos(a) - s.z * std::sin(a), s.y * std::sin(a) + s.z * std::cos(a)};
}
inline Vec3 rot_y(const Vec3& s, double a) {  // :119
    return {s.x * std::cos(a) + s.z * std::sin(a), s.y, s.z * std::cos(a) - s.x * std::sin(a)};
}
inline Vec3 rot_z(const Vec3& s, double a) {  // :127
    return {s.x * std::cos(a) - s.y * std::sin(a), s.x * std::sin(a) + s.y * std::cos(a), s.z};
}
inline double determinant3(const Vec3& v0, const Vec3& v1, const Vec3& v2) {  // :136-140
    return v0.x * (v1.y * v2.z - v1.z * v2.y) - v1.x * (v0.y * v2.z - v0.z * v2.y) +
           v2.x * (v0.y * v1.z - v0.z * v1.y);
}

struct Ray {  // :371-385
    Vec3 pos, dir;
    Vec3 eval(double t) const { return pos + t * dir; }
};

struct Hit {  // :418-424 (+ tri: mesh triangle index, carried for parity checks only)
    double t;
    Vec3 pos, n;
    long id;
    long tri;
    Vec3 dir;  // direction of the ray that made the hit (set by trace_ray; the dielectric needs it behind a mirror)
};

// ---------------------------------------------------------------- Triangle (src/geometry.rs:598-671)
struct Triangle {
    Vec3 a, b, c;
    Vec3 normal() const { return norm(cross(c - a, b - a)); }  // :606-608
    double area() const {                                      // :614-620 Heron
        double ab = mag(a - b), bc = mag(b - c), ca = mag(c - a);
        double s = (ab + bc + ca) / 2.;
        return std::sqrt(s * (s - ab) * (s - bc) * (s - ca));
    }
    Vec3 get_barycentric(double b0, double b1) const {  // :622-628 (does NOT add `a`; kept)
        Vec3 ab = norm(b - a), ac = norm(c - a);
        return ab * b0 + ac * b1;
    }
    bool intersect(const Ray& ray, Hit& out) const {  // :637-670
        Vec3 n = normal();
        if (std::fabs(dot(n, ray.dir)) < 0.0001) return false;
        Vec3 ab = b - a, ac = c - a, bb = ray.pos - a;
        Vec3 md = -ray.dir;
        double det = determinant3(md, ab, ac);
        double t = determinant3(bb, ab, ac) / det;
        double u = determinant3(md, bb, ac) / det;
        double v = determinant3(md, ab, bb) / det;
        if (u < 0. || u > 1. || v < 0. || u + v > 1.) return false;
        if (t > 0.0001) {
            Vec3 nf = dot(n, md) >= 0. ? n : -n;
            out.t = t;
            out.pos = ray.eval(t) + 0.00001 * nf;
            out.n = nf;
            out.id = 10000000;
            return true;
        }
        return false;
    }
};

// ---------------------------------------------------------------- BoundingBox (src/geometry.rs:916-1113)
struct BoundingBox {
    Vec3 min, max;
    static BoundingBox enclose(const std::vector<Vec3>& pts) {  // :927-953
        double inf = std::numeric_limits<double>::infinity();
        BoundingBox b{{inf, inf, inf}, {-inf, -inf, -inf}};
        for (const Vec3& p : pts) {
            if (p.x < b.min.x) b.min.x = p.x;
            if (p.x > b.max.x) b.max.x = p.x;
            if (p.y < b.min.y) b.min.y = p.y;
            if (p.y > b.max.y) b.max.y = p.y;
            if (p.z < b.min.z) b.min.z = p.z;
            if (p.z > b.max.z) b.max.z = p.z;
        }
        return b;
    }
    bool contains(const Vec3& p) const {  // :968-975
        return min.x <= p.x && p.x <= max.x && min.y <= p.y && p.y <= max.y && min.z <= p.z && p.z <= max.z;
    }
    // :977-1036 — first of six faces (L,R,B,T,back,front) with t >= 1e-7 whose hit point lies in
    // the face rectangle; NOT the nearest.  Division by a zero component gives inf/NaN exactly as
    // IEEE does in the reference.
    bool intersect(const Ray& r, double& tout) const {
        const double EPS = 0.0000001;
        double t;
        t = (min.x - r.pos.x) / r.dir.x;
        if (t >= EPS) {
            Vec3 p = r.eval(t);
            if (min.y <= p.y && p.y <= max.y && min.z <= p.z && p.z <= max.z) { tout = t; return true; }
        }
        t = (max.x - r.pos.x) / r.dir.x;
        if (t >= EPS) {
            Vec3 p = r.eval(t);
            if (min.y <= p.y && p.y <= max.y && min.z <= p.z && p.z <= max.z) { tout = t; return true; }
        }
        t = (min.y - r.pos.y) / r.dir.y;
        if (t >= EPS) {
            Vec3 p = r.eval(t);
            if (min.x <= p.x && p.x <= max.x && min.z <= p.z && p.z <= max.z) { tout = t; return true; }
        }
        t = (max.y - r.pos.y) / r.dir.y;
        if (t >= EPS) {
            Vec3 p = r.eval(t);
            if (min.x <= p.x && p.x <= max.x && min.z <= p.z && p.z <= max.z) { tout = t; return true; }
        }
        t = (min.z - r.pos.z) / r.dir.z;
        if (t >= EPS) {
            Vec3 p = r.eval(t);
            if (min.x <= p.x && p.x <= max.x && min.y <= p.y && p.y <= max.y) { tout = t; return true; }
        }
        t = (max.z - r.pos.z) / r.dir.z;
        if (t >= EPS) {
            Vec3 p = r.eval(t);
            if (min.x <= p.x && p.x <= max.x && min.y <= p.y && p.y <= max.y) { tout = t; return true; }
        }
        return false;
    }
    bool intersect_line_segment(const Vec3& a, const Vec3& b) const {  // :1038-1047
        Ray r{a, norm(b - a)};
        double t;
        if (intersect(r, t)) {
            if (t <= mag(b - a)) return true;
        }
        return false;
    }
    bool overlaps_triangle(const Triangle& t) const {  // :1049-1061
        if (contains(t.a) || contains(t.b) || contains(t.c)) return true;
        return intersect_line_segment(t.a, t.b) || intersect_line_segment(t.a, t.c) ||
               intersect_line_segment(t.b, t.c);
    }
    Vec3 center() const { return (min + max) / 2.; }  // :1063-1065
    BoundingBox octant(int i) const {                 // :1067-1099 (bit2 = x, bit1 = y, bit0 = z)
        Vec3 c = center();
        switch (i) {
            case 0: return {min, c};
            case 1: return {V(min.x, min.y, c.z), V(c.x, c.y, max.z)};
            case 2: return {V(min.x, c.y, min.z), V(c.x, max.y, c.z)};
            case 3: return {V(min.x, c.y, c.z), V(c.x, max.y, max.z)};
            case 4: return {V(c.x, min.y, min.z), V(max.x, c.y, c.z)};
            case 5: return {V(c.x, min.y, c.z), V(max.x, c.y, max.z)};
            case 6: return {V(c.x, c.y, min.z), V(max.x, max.y, c.z)};
            default: return {c, max};
        }
    }
};

// ---------------------------------------------------------------- Octree (src/geometry.rs:1133-1301)
struct OctNode {
    bool leaf;
    long children[8];                               // -1 = None
    std::vector<std::pair<long, Triangle>> tris;    // leaf payload (copied, as in the reference)
};

struct Octree {
    std::vector<OctNode> nodes;
    BoundingBox bounding_box;
    static constexpr int MAX_DEPTH = 10;   // :1146
    static constexpr size_t SMALL_NODE = 9;  // :1147

    long build_rec(const BoundingBox& bb, std::vector<std::pair<long, Triangle>> tris, int depth) {  // :1164-1216
        if (tris.empty()) return -1;
        if (tris.size() <= SMALL_NODE || depth >= MAX_DEPTH) {
            OctNode n;
            n.leaf = true;
            n.tris = std::move(tris);
            nodes.push_back(std::move(n));
            return (long)nodes.size() - 1;
        }
        BoundingBox oct[8];
        for (int i = 0; i < 8; ++i) oct[i] = bb.octant(i);
        std::vector<std::pair<long, Triangle>> ot[8];
        for (auto& it : tris)
            for (int i = 0; i < 8; ++i)
                if (oct[i].overlaps_triangle(it.second)) ot[i].push_back(it);
        OctNode n;
        n.leaf = false;
        for (int i = 0; i < 8; ++i) n.children[i] = -1;
        nodes.push_back(n);
        long i_new = (long)nodes.size() - 1;
        long ch[8];
        for (int i = 0; i < 8; ++i) ch[i] = build_rec(oct[i], ot[i], depth + 1);
        for (int i = 0; i < 8; ++i) nodes[i_new].children[i] = ch[i];
        return i_new;
    }

    // :1245-1295.  `work` counts node visits / box tests / triangle tests when non-null.
    bool intersect_rec(const OctNode& node, const BoundingBox& bb, const Ray& ray, Hit& out, long* work) const {
        if (work) work[0]++;
        if (!node.leaf) {
            int order[8] = {0, 1, 2, 3, 4, 5, 6, 7};
            BoundingBox roct[8];
            for (int i = 0; i < 8; ++i) roct[i] = bounding_box.octant(i);  // ROOT's octants (:1249)
            auto dist = [&](int k) { return mag(roct[k].center() - ray.pos); };
            for (int i = 1; i < 8; ++i) {  // insertion sort (:1251-1260)
                int j = i;
                while (j > 0 && dist(order[j - 1]) > dist(order[j])) {
                    std::swap(order[j], order[j - 1]);
                    --j;
                }
            }
            BoundingBox oct[8];
            for (int i = 0; i < 8; ++i) oct[i] = bb.octant(i);
            for (int k = 0; k < 8; ++k) {
                int i = order[k];
                long n = node.children[i];
                if (n >= 0) {
                    double tb;
                    if (work) work[1]++;
                    if (oct[i].intersect(ray, tb)) {
                        if (intersect_rec(nodes[n], oct[i], ray, out, work)) return true;  // early exit (:1267-1270)
                    }
                }
            }
            return false;
        }
        bool found = false;
        Hit best{};
        for (auto& it : node.tris) {  // :1276-1292
            Hit h{};
            if (work) work[2]++;
            if (it.second.intersect(ray, h)) {
                h.tri = it.first;
                if (!found || h.t < best.t) { best = h; found = true; }
            }
        }
        if (found) out = best;
        return found;
    }
    bool intersect(const Ray& ray, Hit& out, long* work) const {  // :1237-1243
        if (nodes.empty()) return false;
        return intersect_rec(nodes[0], bounding_box, ray, out, work);
    }
};

// ---------------------------------------------------------------- exact BVH (oracle-only accelerator for the
// brute-force branch src/geometry.rs:887-903; conservative slab test, so it returns exactly what
// the linear scan returns: minimum t, first triangle index on exact ties).
struct ExactBVH {
    struct Node { double lo[3], hi[3]; int left, right, first, count; };
    std::vector<Node> nodes;
    std::vector<int> order;
    std::vector<Triangle> tris;  // owned copy (objects are moved after the build)

    void build(const std::vector<Triangle>& t) {
        tris = t;
        order.resize(t.size());
        for (size_t i = 0; i < t.size(); ++i) order[i] = (int)i;
        nodes.clear();
        if (!t.empty()) build_rec(0, (int)t.size());
    }
    int build_rec(int first, int count) {
        Node n;
        for (int k = 0; k < 3; ++k) { n.lo[k] = 1e300; n.hi[k] = -1e300; }
        double clo[3] = {1e300, 1e300, 1e300}, chi[3] = {-1e300, -1e300, -1e300};
        for (int i = first; i < first + count; ++i) {
            const Triangle& T = tris[order[i]];
            const Vec3* vs[3] = {&T.a, &T.b, &T.c};
            double c[3] = {0, 0, 0};
            for (auto v : vs) {
                double p[3] = {v->x, v->y, v->z};
                for (int k = 0; k < 3; ++k) { n.lo[k] = std::min(n.lo[k], p[k]); n.hi[k] = std::max(n.hi[k], p[k]); c[k] += p[k] / 3.0; }
            }
            for (int k = 0; k < 3; ++k) { clo[k] = std::min(clo[k], c[k]); chi[k] = std::max(chi[k], c[k]); }
        }
        for (int k = 0; k < 3; ++k) {  // pad: conservative
            double pad = 1e-9 * (1.0 + std::fabs(n.lo[k]) + std::fabs(n.hi[k]));
            n.lo[k] -= pad; n.hi[k] += pad;
        }
        n.left = n.right = -1; n.first = first; n.count = count;
        int idx = (int)nodes.size();
        nodes.push_back(n);
        if (count <= 4) return idx;
        int ax = 0;
        if (chi[1] - clo[1] > chi[ax] - clo[ax]) ax = 1;
        if (chi[2] - clo[2] > chi[ax] - clo[ax]) ax = 2;
        int mid = first + count / 2;
        auto cen = [&](int id) {
            const Triangle& T = tris[id];
            return ax == 0 ? T.a.x + T.b.x + T.c.x : (ax == 1 ? T.a.y + T.b.y + T.c.y : T.a.z + T.b.z + T.c.z);
        };
        std::nth_element(order.begin() + first, order.begin() + mid, order.begin() + first + count,
                         [&](int p, int q) { return cen(p) < cen(q); });
        int l = build_rec(first, mid - first);
        int r = build_rec(mid, first + count - mid);
        nodes[idx].left = l; nodes[idx].right = r; nodes[idx].count = 0;
        return idx;
    }
    static bool slab(const Node& n, const Ray& r, double tmax) {
        double t0 = 0.0, t1 = tmax;
        const double o[3] = {r.pos.x, r.pos.y, r.pos.z}, d[3] = {r.dir.x, r.dir.y, r.dir.z};
        for (int k = 0; k < 3; ++k) {
            if (d[k] == 0.0) {
                if (o[k] < n.lo[k] || o[k] > n.hi[k]) return false;
                continue;
            }
            double inv = 1.0 / d[k];
            double a = (n.lo[k] - o[k]) * inv, b = (n.hi[k] - o[k]) * inv;
            if (a > b) std::swap(a, b);
            a -= 1e-9 * (1.0 + std::fabs(a)); b += 1e-9 * (1.0 + std::fabs(b));
            if (a > t0) t0 = a;
            if (b < t1) t1 = b;
            if (t0 > t1) return false;
        }
        return true;
    }
    bool intersect(const Ray& ray, Hit& out, long* work) const {
        if (nodes.empty()) return false;
        bool found = false;
        Hit best{};
        int stack[128], sp = 0;
        stack[sp++] = 0;
        while (sp) {
            const Node& n = nodes[stack[--sp]];
            if (work) work[0]++;
            double tmax = found ? best.t : std::numeric_limits<double>::infinity();
            if (!slab(n, ray, tmax)) continue;
            if (n.left < 0) {
                for (int i = n.first; i < n.first + n.count; ++i) {
                    Hit h{};
                    if (work) work[2]++;
                    int id = order[i];
                    if (tris[id].intersect(ray, h)) {
                        h.tri = id;
                        // linear scan semantics: strict <, so on exact ties the lowest index wins
                        if (!found || h.t < best.t || (h.t == best.t && id < best.tri)) { best = h; found = true; }
                    }
                }
            } else {
                stack[sp++] = n.left;
                stack[sp++] = n.right;
            }
        }
        if (found) out = best;
        return found;
    }
};

// ---------------------------------------------------------------- Mesh (src/geometry.rs:406-416,753-914)
struct Mesh {
    std::vector<Vec3> vertices;
    std::vector<size_t> indices;
    BoundingBox bounding_box;
    double surface_area = 0;
    std::vector<double> cumulative;  // WeightedIndex cumulative weights (rand 0.8.5 weighted_index.rs)
    Octree octree;
    bool has_octree = false;
    std::vector<Triangle> tri_cache;  // for exact mode
    ExactBVH bvh;

    size_t num_triangles() const { return indices.size() / 3; }
    Triangle triangle(size_t i) const {  // :872-877
        return {vertices[indices[i * 3]], vertices[indices[i * 3 + 1]], vertices[indices[i * 3 + 2]]};
    }
    void init() {  // Mesh::new :754-775
        surface_area = 0;
        cumulative.clear();
        for (size_t i = 0; i < num_triangles(); ++i) {
            surface_area += triangle(i).area();
            cumulative.push_back(surface_area);
        }
        bounding_box = BoundingBox::enclose(vertices);
    }
    Vec3 center() const { return bounding_box.center(); }            // :907
    void fit_bounds() { bounding_box = BoundingBox::enclose(vertices); }  // :911
    void accelerate() {                                                // :835-837, Octree::build :1149-1162
        std::vector<std::pair<long, Triangle>> all;
        for (size_t i = 0; i < num_triangles(); ++i) all.push_back({(long)i, triangle(i)});
        octree.nodes.clear();
        octree.bounding_box = bounding_box;
        octree.build_rec(bounding_box, std::move(all), 1);
        has_octree = true;
        tri_cache.clear();
        for (size_t i = 0; i < num_triangles(); ++i) tri_cache.push_back(triangle(i));
        bvh.build(tri_cache);
    }
};

bool load_obj(const std::string& path, Mesh& m, std::string& err) {  // Mesh::load :777-833
    std::ifstream f(path);
    if (!f) { err = "cannot open " + path; return false; }
    std::string line;
    while (std::getline(f, line)) {
        std::istringstream ss(line);
        std::string cmd;
        if (!(ss >> cmd)) continue;
        if (cmd == "v") {
            double x, y, z;
            if (!(ss >> x >> y >> z)) { err = "ill-formed vertex: " + line; return false; }
            m.vertices.push_back({x, y, z});
        } else if (cmd == "f") {
            for (int k = 0; k < 3; ++k) {
                std::string tok;
                if (!(ss >> tok)) { err = "unexpected end of file"; return false; }
                std::string first = tok.substr(0, tok.find('/'));  // parse_face :708-729 keeps i0 only
                char* end = nullptr;
                long long v = std::strtoll(first.c_str(), &end, 10);
                if (first.empty() || *end != 0 || v < 1) { err = "Ill-formed integer " + first; return false; }
                m.indices.push_back((size_t)(v - 1));
            }
        }  // "vn" is parsed by the reference but never used for shading (:792-797)
    }
    for (size_t i : m.indices)
        if (i >= m.vertices.size()) { err = "face index out of range"; return false; }
    m.init();
    return true;
}

Mesh make_prism(const Vec3& p, double w, double h, double d) {  // :839-862
    Mesh m;
    m.vertices = {V(p.x, p.y, p.z),         V(p.x, p.y, p.z + d),         V(p.x, p.y + h, p.z),
                  V(p.x, p.y + h, p.z + d), V(p.x + w, p.y, p.z),         V(p.x + w, p.y, p.z + d),
                  V(p.x + w, p.y + h, p.z), V(p.x + w, p.y + h, p.z + d)};
    m.indices = {1, 3, 7, 1, 5, 7, 0, 2, 6, 0, 4, 6, 0, 1, 3, 0, 2, 3,
                 4, 5, 7, 4, 6, 7, 2, 3, 7, 2, 6, 7, 0, 1, 5, 0, 4, 5};
    m.init();
    return m;
}

// ---------------------------------------------------------------- Geometry / Object / BRDF
enum GeomKind { G_SPHERE = 0, G_PLANE = 1, G_MESH = 2 };
enum BrdfKind { B_DIFFUSE = 0, B_SPECULAR = 1, B_PHONG = 2, B_DIELECTRIC = 3 };

struct BRDF {  // src/scene.rs:17-28
    int kind;
    Vec3 k;  // kd (Diffuse) or ks (Specular); Dielectric: {ior, orientation sign, 0}, tint in color_d
    double kd, ks;
    int power;
    Vec3 color_d, color_s;
};

struct Object {  // src/scene.rs:10-15
    Vec3 emitted;
    BRDF brdf;
    int gkind;
    Vec3 pos;  // sphere centre / plane point
    double r;
    Vec3 n;    // plane normal
    Mesh mesh;
};

// ---------------------------------------------------------------- Philox4x32-10 (Salmon, Moraes, Dror, Shaw, SC'11)
struct Philox {
    static inline void round(uint32_t c[4], uint32_t k0, uint32_t k1) {
        uint64_t p0 = (uint64_t)0xD2511F53u * c[0];
        uint64_t p1 = (uint64_t)0xCD9E8D57u * c[2];
        uint32_t n0 = (uint32_t)(p1 >> 32) ^ c[1] ^ k0;
        uint32_t n1 = (uint32_t)p1;
        uint32_t n2 = (uint32_t)(p0 >> 32) ^ c[3] ^ k1;
        uint32_t n3 = (uint32_t)p0;
        c[0] = n0; c[1] = n1; c[2] = n2; c[3] = n3;
    }
    static inline void gen(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1, uint32_t out[4]) {
        uint32_t c[4] = {c0, c1, c2, c3};
        for (int i = 0; i < 10; ++i) {
            round(c, k0, k1);
            k0 += 0x9E3779B9u;
            k1 += 0xBB67AE85u;
        }
        out[0] = c[0]; out[1] = c[1]; out[2] = c[2]; out[3] = c[3];
    }
};
// uniform in (0,1): 24 bits, centred — the same value the fp32 CUDA path uses
inline double u01(uint32_t x) { return ((double)(x >> 8) + 0.5) * (1.0 / 16777216.0); }

inline double u24(uint32_t v) { return ((double)v + 0.5) * (1.0 / 16777216.0); }

struct Sampler {  // RNG contract (DESIGN.md): counter = (pixel, sample, depth, block), key = seed
    uint32_t pixel, sample, k0, k1;
    void block(uint32_t depth, uint32_t blk, double u[4]) const {
        uint32_t o[4];
        Philox::gen(pixel, sample, depth, blk, k0, k1, o);
        for (int i = 0; i < 4; ++i) u[i] = u01(o[i]);
    }
    // live vertex: ONE Philox block -> {light u1, light u2, russian roulette, brdf u1, brdf u2}
    void vertex(uint32_t depth, double u[5]) const {
        uint32_t o[4];
        Philox::gen(pixel, sample, depth, 0, k0, k1, o);
        u[0] = u24(o[0] >> 8);
        u[1] = u24(o[1] >> 8);
        u[2] = u24(o[2] >> 8);
        u[3] = u24(o[3] >> 8);
        u[4] = u24(((o[0] & 0xffu) << 16) | ((o[1] & 0xffu) << 8) | (o[2] & 0xffu));
    }
};

struct Counters {  // one instance per render thread
    long rays = 0, samples = 0;
};

struct Scene {  // src/scene.rs:101-107
    Ray camera;
    std::vector<Object> objects;
    long light_source = -1;
    int accel = 1;      // 0 octree_faithful, 1 exact
    int estimator = 0;  // 0 NEE live, 1 dead MIS branch
    std::string err;

    // ---- Geometry::intersect  src/geometry.rs:512-571
    bool geom_intersect(const Object& o, const Ray& ray, Hit& out, long* work) const {
        if (o.gkind == G_SPHERE) {
            Vec3 op = o.pos - ray.pos;
            double eps = 1e-4;
            double b = dot(op, ray.dir);
            double det = b * b - dot(op, op) + o.r * o.r;
            if (det < 0.) return false;
            det = std::sqrt(det);
            double t = b - det;
            if (t > eps) {
                Vec3 pos = ray.eval(t);
                Vec3 n = norm(pos - o.pos);
                out = {t, pos, dot(n, -ray.dir) >= 0. ? n : -n, 1000000, -1};
                return true;
            }
            t = b + det;
            if (t > eps) {
                Vec3 pos = ray.eval(t);
                Vec3 n = norm(pos - o.pos);
                out = {t, pos, dot(n, -ray.dir) >= 0. ? n : -n, 1000000, -1};
                return true;
            }
            return false;
        }
        if (o.gkind == G_PLANE) {
            double d_dot_n = dot(ray.dir, o.n);
            if (std::fabs(d_dot_n) < 0.0001) return false;
            double t = dot(o.pos - ray.pos, o.n) / dot(ray.dir, o.n);
            if (t >= 0.) {
                Vec3 n = dot(o.n, -ray.dir) >= 0. ? o.n : -o.n;
                out = {t, ray.eval(t) + n * 0.00001, n, 1000000, -1};
                return true;
            }
            return false;
        }
        // Mesh::intersect :883-905
        if (accel == 0) return o.mesh.octree.intersect(ray, out, work);
        return o.mesh.bvh.intersect(ray, out, work);
    }

    // ---- Scene::trace_ray  src/scene.rs:272-289 (strict <: lowest object index wins ties)
    bool trace_ray(const Ray& ray, Hit& nearest, Counters* cnt, long* work = nullptr) const {
        if (cnt) cnt->rays++;
        bool found = false;
        for (size_t i = 0; i < objects.size(); ++i) {
            Hit h{};
            if (geom_intersect(objects[i], ray, h, work)) {
                h.id = (long)i;
                if (!found || h.t < nearest.t) { nearest = h; found = true; }
            }
        }
        if (found) nearest.dir = ray.dir;
        return found;
    }

    // ---- create_local_coord  src/scene.rs:112-123
    static void create_local_coord(const Vec3& n, Vec3& u, Vec3& v, Vec3& w) {
        w = n;
        u = norm(cross(std::fabs(w.x) > 0.1 ? V(0., 1., 0.) : V(1., 0., 0.), w));
        v = cross(w, u);
    }

    // ---- BRDF::eval  src/scene.rs:31-54
    static Vec3 brdf_eval(const BRDF& f, const Vec3& n, const Vec3& o, const Vec3& i) {
        switch (f.kind) {
            case B_DIFFUSE: return f.k * FRAC_1_PI;
            case B_SPECULAR:
                if (equal_within(i, flip_across(o, n), 0.001)) return f.k / dot(n, i);
                return V(0, 0, 0);
            default: {
                Vec3 reflection = flip_across(i, n);
                double c = std::max(dot(o, reflection), (double)0.);
                double pw = 1.0;  // powi
                for (int k = 0; k < f.power; ++k) pw *= c;
                return f.color_d * f.kd * FRAC_1_PI + f.color_s * f.ks * (double)(f.power + 2) / (2. * PI) * pw;
            }
        }
    }

    // ---- BRDF::sample_incoming  src/scene.rs:56-98.  xi = {u1, u2, lobe}
    static void brdf_sample(const BRDF& f, const Vec3& n, const Vec3& o, const double xi[4], Vec3& i, double& pdf) {
        switch (f.kind) {
            case B_DIFFUSE: {
                double z = std::sqrt(xi[0]);
                double r = std::sqrt(1.0 - z * z);
                double phi = 2.0 * PI * xi[1];
                double x = r * std::cos(phi), y = r * std::sin(phi);
                Vec3 u, v, w;
                create_local_coord(n, u, v, w);
                i = norm(u * x + v * y + w * z);
                pdf = dot(n, i) * FRAC_1_PI;
                return;
            }
            case B_SPECULAR:
                i = flip_across(o, n);
                pdf = 1.0;
                return;
            default: {
                double p = (double)f.power;
                double u = xi[2];
                if (u < f.kd) {  // local coordinates, never rotated into the n frame (reference quirk)
                    double xi1 = xi[0], xi2 = xi[1];
                    i = V(std::sqrt(1. - xi1) * std::cos(2. * PI * xi2), std::sqrt(1. - xi1) * std::sin(2. * PI * xi2),
                          std::sqrt(xi1));
                    pdf = dot(n, i) * FRAC_1_PI;
                } else if (f.kd <= u && u < f.kd + f.ks) {
                    double xi1 = xi[0], xi2 = xi[1];
                    double s = std::sqrt(1. - std::pow(xi1, 2. / (p + 1.)));
                    i = V(s * std::cos(2. * PI * xi2), s * std::sin(2. * PI * xi2), std::pow(xi1, 1. / (p + 1.)));
                    double pw = 1.0;
                    for (int k = 0; k < f.power; ++k) pw *= i.z;
                    pdf = (p + 1.) / (2. * PI) * pw;
                } else {
                    i = V(0, 0, 0);
                    pdf = 1.0;
                }
            }
        }
    }

    // ---- Geometry::sample  src/geometry.rs:573-595.  xi = {u1, u2, -, select}
    bool light_sample(const double xi[4], Vec3& y, Vec3& ny, double& pdf) const {
        const Object& L = objects[light_source];
        if (L.gkind == G_SPHERE) {
            double z = 2. * xi[0] - 1.;
            double x = std::sqrt(1.0 - z * z) * std::cos(2. * PI * xi[1]);
            double yy = std::sqrt(1.0 - z * z) * std::sin(2. * PI * xi[1]);
            Vec3 n = norm(V(x, yy, z));
            y = L.pos + n * L.r;
            ny = n;
            pdf = 1.0 / (4.0 * PI * L.r * L.r);
            return true;
        }
        if (L.gkind == G_MESH) {
            // WeightedIndex<f64>::sample (rand 0.8.5): chosen = U[0,total); partition_point(w <= chosen)
            const Mesh& m = L.mesh;
            double chosen = xi[3] * m.surface_area;
            size_t idx = std::upper_bound(m.cumulative.begin(), m.cumulative.end(), chosen) - m.cumulative.begin();
            if (idx >= m.num_triangles()) idx = m.num_triangles() - 1;
            Triangle t = m.triangle(idx);
            double b0 = 1. - std::sqrt(xi[0]);  // Triangle::sample :630-635
            double b1 = (1. - b0) * xi[1];
            y = t.get_barycentric(b0, b1);
            ny = t.normal();
            pdf = 1. / m.surface_area;
            return true;
        }
        return false;  // Plane: unimplemented!() :593
    }

    // ---- mutually_visible  src/scene.rs:258-270
    bool mutually_visible(const Vec3& x, const Vec3& y, Counters* cnt) const {
        const double ERR_MARGIN = 0.001;
        Vec3 diff = y - x;
        Ray r{x, norm(diff)};
        Hit h{};
        if (trace_ray(r, h, cnt)) return h.t + ERR_MARGIN >= mag(diff);
        return true;
    }

    // ---- reflected_radiance  src/scene.rs:161-244
    Vec3 reflected_radiance(const Hit& hit, const Vec3& o, uint64_t depth, const Sampler& s, Counters* cnt) const {
        const Vec3& x = hit.pos;
        const Vec3& n = hit.n;
        const Object& obj = objects[hit.id];
        double p = depth <= 5 ? 1.0 : 0.9;  // MAX_BOUNCES / SURVIVAL_PROBABILITY :109-110,164-168
        double v5[5], sel[4];
        s.vertex((uint32_t)depth, v5);     // {light u1, light u2, RR, brdf u1, brdf u2}
        s.block((uint32_t)depth, 1, sel);  // {phong lobe select, light triangle select, -, -}
        const double b0[4] = {v5[0], v5[1], v5[2], sel[1]};  // light sample + roulette
        const double b1[4] = {v5[3], v5[4], sel[0], 0.0};    // continuation BRDF sample

        if (obj.brdf.kind == B_DIELECTRIC) {  // smooth glass, DESIGN §3e
            Vec3 rad = V(0, 0, 0);
            if (b0[2] < p) {
                const Vec3 d = hit.dir;  // the true direction (a mirror in front hands the recursion a stale `o`)
                bool flipped;            // did the ray meet the side the stored normal points away from?
                if (obj.gkind == G_SPHERE) flipped = dot(n, x - obj.pos) < 0.;
                else if (obj.gkind == G_PLANE) flipped = dot(n, obj.n) < 0.;
                else flipped = dot(n, obj.mesh.triangle((size_t)hit.tri).normal()) < 0.;
                const bool entering = !flipped != (obj.brdf.k.y < 0.);
                const double ior = obj.brdf.k.x, eta = entering ? 1. / ior : ior;
                const double cos_i = -dot(d, n), sin2t = eta * eta * (1. - cos_i * cos_i);
                double F = 1., cos_t = 0.;
                if (sin2t < 1.) {
                    cos_t = std::sqrt(1. - sin2t);
                    const double rs = (eta * cos_i - cos_t) / (eta * cos_i + cos_t);
                    const double rp = (cos_i - eta * cos_t) / (cos_i + eta * cos_t);
                    F = 0.5 * (rs * rs + rp * rp);
                }
                Vec3 org = x, i, w = V(1, 1, 1);
                if (b1[0] < F) {
                    i = d + 2. * cos_i * n;
                } else {  // through the surface: planes and triangles start 1e-5 behind it, spheres on it
                    i = eta * d + (eta * cos_i - cos_t) * n;
                    if (obj.gkind != G_SPHERE) org = x - 0.00002 * n;
                    w = obj.brdf.color_d;
                }
                Hit h2{};
                if (trace_ray(Ray{org, i}, h2, cnt))
                    rad = mult(objects[h2.id].emitted + reflected_radiance(h2, -i, depth + 1, s, cnt), w) / p;
            }
            return rad;
        }
        if (obj.brdf.kind == B_SPECULAR) {  // :170-185
            Vec3 rad = V(0, 0, 0);
            if (b0[2] < p) {
                Vec3 i;
                double pdf;
                brdf_sample(obj.brdf, n, o, b1, i, pdf);
                Hit h2{};
                if (trace_ray(Ray{x, i}, h2, cnt)) {
                    // emitted + (R ⊙ f) * (n·i) / (pdf*p); NOTE: recursion gets `o`, not -i (:178)
                    rad = objects[h2.id].emitted +
                          mult(reflected_radiance(h2, o, depth + 1, s, cnt), brdf_eval(obj.brdf, n, o, i)) * dot(n, i) /
                              (pdf * p);
                }
            }
            return rad;
        }

        Vec3 rad;
        if (estimator == 1) {  // dead branch :189-216, verbatim (fresh-sample pdfs included)
            Vec3 rad_direct = V(0, 0, 0);
            double b2[4], b3[4], b4[4];
            s.block((uint32_t)depth, 2, b2);  // fresh BRDF sample used only for its pdf (:195)
            s.block((uint32_t)depth, 3, b3);  // second light point (:206)
            s.block((uint32_t)depth, 4, b4);  // this branch's own BRDF sample (:203), independent of the continuation's
            Vec3 y, ny;
            double pdf_light;
            light_sample(b0, y, ny, pdf_light);
            Vec3 i = norm(y - x);
            if (mutually_visible(x, y, cnt)) {
                pdf_light *= dot(y - x, y - x) / dot(ny, -i);
                Vec3 itmp;
                double pdf_brdf;
                brdf_sample(obj.brdf, n, i, b2, itmp, pdf_brdf);
                rad_direct += mult(objects[light_source].emitted, brdf_eval(obj.brdf, n, o, i)) * dot(n, i) /
                              (pdf_light + pdf_brdf);
            }
            Vec3 i2;
            double pdf_brdf2;
            brdf_sample(obj.brdf, n, o, b4, i2, pdf_brdf2);
            Hit h2{};
            if (trace_ray(Ray{x, i2}, h2, cnt)) {
                if (h2.id == light_source) {
                    Vec3 y2, ny2;
                    double pdf_light2;
                    light_sample(b3, y2, ny2, pdf_light2);
                    pdf_light2 *= dot(y2 - x, y2 - x) / dot(ny2, -i2);
                    rad_direct += mult(objects[light_source].emitted, brdf_eval(obj.brdf, n, o, i2)) * dot(n, i2) /
                                  (pdf_brdf2 + pdf_light2);
                }
            }
            rad = rad_direct;
        } else {  // live NEE :217-229
            Vec3 y, ny;
            double pdf;
            light_sample(b0, y, ny, pdf);
            Vec3 i = norm(y - x);
            double r_sqr = dot(y - x, y - x);
            double visibility = mutually_visible(x, y, cnt) ? 1. : 0.;
            rad = mult(objects[light_source].emitted, brdf_eval(obj.brdf, n, o, i)) * visibility * dot(n, i) *
                  dot(ny, -i) / (r_sqr * pdf);
        }

        if (b0[2] < p) {  // :231-240
            Vec3 i;
            double pdf_brdf;
            brdf_sample(obj.brdf, n, o, b1, i, pdf_brdf);
            Hit h2{};
            if (trace_ray(Ray{x, i}, h2, cnt)) {
                rad += mult(reflected_radiance(h2, -i, depth + 1, s, cnt), brdf_eval(obj.brdf, n, o, i)) * dot(n, i) /
                       (pdf_brdf * p);
            }
        }
        return rad;
    }

    // ---- received_radiance  src/scene.rs:152-159
    Vec3 received_radiance(const Ray& r, const Sampler& s, Counters* cnt) const {
        Hit hit{};
        if (cnt) cnt->samples++;
        if (trace_ray(r, hit, cnt)) return objects[hit.id].emitted + reflected_radiance(hit, -r.dir, 1, s, cnt);
        return V(0, 0, 0);
    }
};

// camera basis  src/server.rs:328-331
inline void camera_basis(const Scene& sc, int width, int height, Vec3& cx, Vec3& cy) {
    double w = (double)width, h = (double)height;
    cx = V(w * 0.5135 / h, 0., 0.);
    cy = norm(cross(cx, sc.camera.dir)) * 0.5135;
}
// camera ray for sub-pixel (sx,sy) with jitter (dx,dy); y is the sampler's (bottom-up) row. :353-357
inline Ray camera_ray(const Scene& sc, const Vec3& cx, const Vec3& cy, int x, int y, int width, int height, int sx,
                      int sy, double dx, double dy) {
    double w = (double)width, h = (double)height;
    Vec3 d = cx * ((((double)sx + 0.5 + dx) / 2. + (double)x) / w - 0.5) +
             cy * ((((double)sy + 0.5 + dy) / 2. + (double)y) / h - 0.5) + sc.camera.dir;
    return Ray{sc.camera.pos, norm(d)};
}
inline double tent(double u) {  // :339-344
    double r = 2. * u;
    return r < 1. ? std::sqrt(r) - 1. : 1. - std::sqrt(2. - r);
}

// sample_pixel  src/server.rs:320-364.  y_img is the top-down screen row (message row);
// the sampler's own y is height - y_img - 1 (:181).  `sub` (optional) receives the four
// un-clamped sub-pixel means (order sy*2+sx, rgb).
Vec3 sample_pixel(const Scene& sc, int x, int y_img, int width, int height, int spp, uint64_t seed, Counters* cnt,
                  double* sub) {
    int y = height - y_img - 1;
    Vec3 cx, cy;
    camera_basis(sc, width, height, cx, cy);
    int num_samples = spp / 4;
    Vec3 pixel = V(0, 0, 0);
    Sampler s;
    s.pixel = (uint32_t)(y_img * width + x);
    s.k0 = (uint32_t)seed;
    s.k1 = (uint32_t)(seed >> 32);
    for (int sy = 0; sy < 2; ++sy)
        for (int sx = 0; sx < 2; ++sx) {
            Vec3 rad = V(0, 0, 0);
            for (int k = 0; k < num_samples; ++k) {
                s.sample = (uint32_t)((sy * 2 + sx) * num_samples + k);
                double u[4];
                s.block(0, 0, u);
                double dx = tent(u[0]), dy = tent(u[1]);
                Ray r = camera_ray(sc, cx, cy, x, y, width, height, sx, sy, dx, dy);
                rad += sc.received_radiance(r, s, cnt) * (1. / (double)num_samples);
            }
            if (sub) {
                double* q = sub + (sy * 2 + sx) * 3;
                q[0] = rad.x; q[1] = rad.y; q[2] = rad.z;
            }
            pixel += clampv(rad, 0., 1.) * 0.25;
        }
    // gamma_correct :366-368
    Vec3 c = clampv(pixel, 0., 1.);
    return V(std::pow(c.x, 1.0 / 2.2) * 255.0 + 0.5, std::pow(c.y, 1.0 / 2.2) * 255.0 + 0.5,
             std::pow(c.z, 1.0 / 2.2) * 255.0 + 0.5);
}

inline uint8_t as_u8(double v) {  // Rust `as u8`: truncate, saturate, NaN -> 0
    if (!(v == v)) return 0;
    if (v <= 0.) return 0;
    if (v >= 255.) return 255;
    return (uint8_t)v;
}

// A dielectric mesh has one orientation sign: whether the stored normal of its first triangle points out of the solid.
// Each connected piece (triangles joined by edges between equal vertex positions) is wound consistently, starting from
// its lowest triangle, and oriented by its signed volume; triangles wound against the first one are turned around.
double orient_dielectric(Mesh& m) {
    const size_t n = m.num_triangles();
    std::map<std::tuple<double, double, double>, long> ids;
    std::vector<long> vid(3 * n);
    for (size_t k = 0; k < 3 * n; ++k) {
        const Vec3& p = m.vertices[m.indices[k]];
        auto it = ids.find({p.x, p.y, p.z});
        if (it == ids.end()) it = ids.insert({{p.x, p.y, p.z}, (long)ids.size()}).first;
        vid[k] = it->second;
    }
    std::map<std::pair<long, long>, std::vector<size_t>> by_edge;
    auto edge = [&](size_t t, int e) { return std::make_pair(vid[3 * t + e], vid[3 * t + (e + 1) % 3]); };
    for (size_t t = 0; t < n; ++t)
        for (int e = 0; e < 3; ++e) {
            auto [a, b] = edge(t, e);
            if (a != b) by_edge[{std::min(a, b), std::max(a, b)}].push_back(t);
        }
    std::vector<int> same(n, 0), outward(n, 1);  // same: +1 wound like the piece's first triangle, -1 against it
    for (size_t first = 0; first < n; ++first) {
        if (same[first]) continue;
        same[first] = 1;
        std::vector<size_t> piece{first};
        double six_vol = 0;
        for (size_t q = 0; q < piece.size(); ++q) {
            const size_t t = piece[q];
            const Triangle tr = m.triangle(t);
            six_vol += same[t] * dot(tr.a, cross(tr.b, tr.c));
            for (int e = 0; e < 3; ++e) {
                auto [a, b] = edge(t, e);
                if (a == b) continue;
                for (size_t u : by_edge[{std::min(a, b), std::max(a, b)}]) {
                    if (same[u]) continue;
                    bool along = false;  // does u run through the edge in the same direction as t?
                    for (int f = 0; f < 3; ++f) along = along || edge(u, f) == std::make_pair(a, b);
                    same[u] = along ? -same[t] : same[t];
                    piece.push_back(u);
                }
            }
        }
        // positive volume: the piece's winding is counter-clockwise seen from outside, (b-a) x (c-a) points out, and the
        // stored normal (c-a) x (b-a) of a triangle wound that way points in
        for (size_t t : piece) outward[t] = six_vol > 0 ? -same[t] : same[t];
    }
    for (size_t t = 0; t < n; ++t)
        if (outward[t] != outward[0]) std::swap(m.indices[3 * t + 1], m.indices[3 * t + 2]);
    return (double)outward[0];
}

}  // namespace

// =============================================================================== C ABI (ctypes)
extern "C" {

void* or_scene_new(const double* cam_pos, const double* cam_dir) {
    Scene* s = new Scene();
    s->camera = Ray{V(cam_pos[0], cam_pos[1], cam_pos[2]), V(cam_dir[0], cam_dir[1], cam_dir[2])};
    return s;
}
void or_scene_free(void* p) { delete (Scene*)p; }
const char* or_last_error(void* p) { return ((Scene*)p)->err.c_str(); }

// brdf: kind, params = Diffuse{kd[3]} | Specular{ks[3]} | Phong{kd,ks,power,color_d[3],color_s[3]} | Dielectric{ior,tint[3]}
// geom: kind 0 sphere {pos[3], r}; 1 plane {pos[3], n[3]}; 2 mesh file; 3 prism {pos[3], size[3]}
// transforms (src/scene.rs:411-429): kind 0 translate[3], 1 scale, 2 rotate_x, 3 rotate_y, 4 rotate_z
int or_add_object(void* sp, const double* emitted, int brdf_kind, const double* bp, int geom_kind, const double* gp,
                  const char* mesh_path, int n_tr, const int* tr_kind, const double* tr_val) {
    Scene* s = (Scene*)sp;
    Object o;
    o.emitted = V(emitted[0], emitted[1], emitted[2]);
    o.brdf = BRDF{};
    o.brdf.kind = brdf_kind;
    if (brdf_kind == B_PHONG) {
        o.brdf.kd = bp[0]; o.brdf.ks = bp[1]; o.brdf.power = (int)bp[2];
        o.brdf.color_d = V(bp[3], bp[4], bp[5]);
        o.brdf.color_s = V(bp[6], bp[7], bp[8]);
    } else if (brdf_kind == B_DIELECTRIC) {
        o.brdf.k = V(bp[0], 1, 0);
        o.brdf.color_d = V(bp[1], bp[2], bp[3]);
    } else {
        o.brdf.k = V(bp[0], bp[1], bp[2]);
    }
    o.r = 0; o.pos = V(0, 0, 0); o.n = V(0, 0, 0);
    if (geom_kind == 0) { o.gkind = G_SPHERE; o.pos = V(gp[0], gp[1], gp[2]); o.r = gp[3]; }
    else if (geom_kind == 1) { o.gkind = G_PLANE; o.pos = V(gp[0], gp[1], gp[2]); o.n = V(gp[3], gp[4], gp[5]); }
    else if (geom_kind == 2) {
        o.gkind = G_MESH;
        if (!load_obj(mesh_path, o.mesh, s->err)) return -3;
    } else { o.gkind = G_MESH; o.mesh = make_prism(V(gp[0], gp[1], gp[2]), gp[3], gp[4], gp[5]); }

    for (int k = 0; k < n_tr; ++k) {  // Geometry::{translate,scale,rotate_*}  src/geometry.rs:427-510
        const double* v = tr_val + 3 * k;
        switch (tr_kind[k]) {
            case 0: {
                Vec3 t = V(v[0], v[1], v[2]);
                if (o.gkind == G_MESH) {
                    for (auto& p : o.mesh.vertices) p += t;
                    o.mesh.bounding_box.min += t;
                    o.mesh.bounding_box.max += t;
                } else o.pos += t;
                break;
            }
            case 1: {
                double sc = v[0];
                if (o.gkind == G_SPHERE) o.r *= sc;
                else if (o.gkind == G_MESH) {
                    Vec3 c = o.mesh.center();
                    for (auto& p : o.mesh.vertices) p = c + (p - c) * sc;
                    // reference quirk (:503-506): min + (min-c)*s, not c + (min-c)*s
                    o.mesh.bounding_box.min = o.mesh.bounding_box.min + (o.mesh.bounding_box.min - c) * sc;
                    o.mesh.bounding_box.max = o.mesh.bounding_box.max + (o.mesh.bounding_box.max - c) * sc;
                }
                break;
            }
            case 2: case 3: case 4: {
                double a = v[0];
                auto rot = [&](const Vec3& q) { return tr_kind[k] == 2 ? rot_x(q, a) : (tr_kind[k] == 3 ? rot_y(q, a) : rot_z(q, a)); };
                if (o.gkind == G_PLANE) o.n = rot(o.n);
                else if (o.gkind == G_MESH) {
                    Vec3 c = o.mesh.center();
                    for (auto& p : o.mesh.vertices) p = c + rot(p - c);
                    o.mesh.fit_bounds();
                }
                break;
            }
            default: s->err = "bad transform"; return -2;
        }
    }
    if (o.gkind == G_MESH && brdf_kind == B_DIELECTRIC) o.brdf.k.y = orient_dielectric(o.mesh);
    if (o.gkind == G_MESH) {
        // NOTE: Mesh::new computed surface areas before the transforms and never refreshes them
        // (src/geometry.rs:755-775); kept: area tables stay those of the untransformed mesh.
        o.mesh.accelerate();
    }
    s->objects.push_back(std::move(o));
    return 0;
}

// Scene::new  src/scene.rs:126-141 — first object whose emitted differs from 0 by >= 1e-5.
long or_scene_finish(void* sp) {
    Scene* s = (Scene*)sp;
    s->light_source = -1;
    for (size_t i = 0; i < s->objects.size(); ++i)
        if (!equal_within(s->objects[i].emitted, V(0, 0, 0), 0.00001)) { s->light_source = (long)i; break; }
    return s->light_source;
}

void or_set_modes(void* sp, int accel, int estimator) {
    Scene* s = (Scene*)sp;
    s->accel = accel;
    s->estimator = estimator;
}

long or_num_objects(void* sp) { return (long)((Scene*)sp)->objects.size(); }
long or_mesh_stats(void* sp, long obj, double* bbox6, long* counts4) {
    Scene* s = (Scene*)sp;
    const Object& o = s->objects[obj];
    if (o.gkind != G_MESH) return -1;
    const BoundingBox& b = o.mesh.bounding_box;
    bbox6[0] = b.min.x; bbox6[1] = b.min.y; bbox6[2] = b.min.z;
    bbox6[3] = b.max.x; bbox6[4] = b.max.y; bbox6[5] = b.max.z;
    long parents = 0, leaves = 0, refs = 0;
    for (auto& n : o.mesh.octree.nodes) {
        if (n.leaf) { leaves++; refs += (long)n.tris.size(); } else parents++;
    }
    counts4[0] = (long)o.mesh.num_triangles(); counts4[1] = parents; counts4[2] = leaves; counts4[3] = refs;
    return 0;
}
// transformed mesh vertices (for cross-checking the product loader): returns n_tris, writes 9 doubles / tri
long or_mesh_triangles(void* sp, long obj, double* out, long cap) {
    Scene* s = (Scene*)sp;
    const Object& o = s->objects[obj];
    if (o.gkind != G_MESH) return -1;
    long n = (long)o.mesh.num_triangles();
    for (long i = 0; i < n && i < cap; ++i) {
        Triangle t = o.mesh.triangle(i);
        double* q = out + 9 * i;
        q[0] = t.a.x; q[1] = t.a.y; q[2] = t.a.z; q[3] = t.b.x; q[4] = t.b.y; q[5] = t.b.z; q[6] = t.c.x; q[7] = t.c.y; q[8] = t.c.z;
    }
    return n;
}

// BoundingBox::octants (the reference's one unit test, src/geometry.rs:1115-1131)
void or_octants(const double* mn, const double* mx, double* out48) {
    BoundingBox b{V(mn[0], mn[1], mn[2]), V(mx[0], mx[1], mx[2])};
    for (int i = 0; i < 8; ++i) {
        BoundingBox o = b.octant(i);
        double* q = out48 + 6 * i;
        q[0] = o.min.x; q[1] = o.min.y; q[2] = o.min.z; q[3] = o.max.x; q[4] = o.max.y; q[5] = o.max.z;
    }
}

// trace_ray on caller-supplied rays.  obj = -1 on miss.  pos/nrm optional (3 doubles each).
void or_trace_rays(void* sp, long n, const double* org, const double* dir, int32_t* obj, int32_t* tri, double* t,
                   double* pos, double* nrm, long* work3) {
    Scene* s = (Scene*)sp;
    for (long i = 0; i < n; ++i) {
        Ray r{V(org[3 * i], org[3 * i + 1], org[3 * i + 2]), V(dir[3 * i], dir[3 * i + 1], dir[3 * i + 2])};
        Hit h{};
        if (s->trace_ray(r, h, nullptr, work3)) {
            obj[i] = (int32_t)h.id;
            tri[i] = s->objects[h.id].gkind == G_MESH ? (int32_t)h.tri : -1;
            t[i] = h.t;
            if (pos) { pos[3 * i] = h.pos.x; pos[3 * i + 1] = h.pos.y; pos[3 * i + 2] = h.pos.z; }
            if (nrm) { nrm[3 * i] = h.n.x; nrm[3 * i + 1] = h.n.y; nrm[3 * i + 2] = h.n.z; }
        } else {
            obj[i] = -1; tri[i] = -1; t[i] = std::numeric_limits<double>::infinity();
        }
    }
}

// camera rays for every pixel at a fixed sub-pixel (sx,sy) and jitter (dx,dy); row 0 = top.
void or_primary_rays(void* sp, int width, int height, int sx, int sy, double dx, double dy, double* org, double* dir) {
    Scene* s = (Scene*)sp;
    Vec3 cx, cy;
    camera_basis(*s, width, height, cx, cy);
    for (int yi = 0; yi < height; ++yi)
        for (int x = 0; x < width; ++x) {
            Ray r = camera_ray(*s, cx, cy, x, height - yi - 1, width, height, sx, sy, dx, dy);
            long i = (long)yi * width + x;
            org[3 * i] = r.pos.x; org[3 * i + 1] = r.pos.y; org[3 * i + 2] = r.pos.z;
            dir[3 * i] = r.dir.x; dir[3 * i + 1] = r.dir.y; dir[3 * i + 2] = r.dir.z;
        }
}

// Render rows [y0,y1) (top-down) of a width x height frame.  rgb8 (h*w*3, optional) gets the
// bytes RenderJob::run would send (src/server.rs:187-189); sub (h*w*12 doubles, optional) the
// un-clamped sub-pixel means.  Threads split the row range into bands like src/server.rs:166-168.
// counters2 = {rays, samples}.
void or_render(void* sp, int width, int height, int spp, uint64_t seed, int y0, int y1, int row_stride, int nthreads,
               uint8_t* rgb8, double* sub, long* counters2) {
    Scene* s = (Scene*)sp;
    // nthreads > 0: static row bands exactly like src/server.rs:166-168;
    // nthreads < 0: |nthreads| threads pulling rows from a shared counter (test convenience only).
    bool dynamic = nthreads < 0;
    if (dynamic) nthreads = -nthreads;
    if (nthreads < 1) nthreads = 1;
    if (row_stride < 1) row_stride = 1;
    int rows = (y1 - y0 + row_stride - 1) / row_stride;  // rows y0, y0+stride, ... < y1
    std::vector<Counters> cnts((size_t)nthreads);
    std::atomic<int> next_row{0};
    auto do_row = [&](int y, Counters* cnt) {
        for (int x = 0; x < width; ++x) {
            long i = (long)y * width + x;
            Vec3 c = sample_pixel(*s, x, y, width, height, spp, seed, cnt, sub ? sub + 12 * i : nullptr);
            if (rgb8) { rgb8[3 * i] = as_u8(c.x); rgb8[3 * i + 1] = as_u8(c.y); rgb8[3 * i + 2] = as_u8(c.z); }
        }
    };
    auto band = [&](int t) {
        if (dynamic) {
            for (int j = next_row.fetch_add(1); j < rows; j = next_row.fetch_add(1)) do_row(y0 + j * row_stride, &cnts[t]);
        } else {
            for (int j = t * rows / nthreads; j < (t + 1) * rows / nthreads; ++j) do_row(y0 + j * row_stride, &cnts[t]);
        }
    };
    if (nthreads == 1) band(0);
    else {
        std::vector<std::thread> th;
        for (int t = 0; t < nthreads; ++t) th.emplace_back(band, t);
        for (auto& t : th) t.join();
    }
    if (counters2) {
        counters2[0] = counters2[1] = 0;
        for (auto& c : cnts) { counters2[0] += c.rays; counters2[1] += c.samples; }
    }
}

// One sample's radiance for an explicit (pixel, sample) — path-level parity probe.
void or_sample_radiance(void* sp, int width, int height, int spp, uint64_t seed, long n, const int32_t* px,
                        const int32_t* py_img, const int32_t* sample_idx, double* rgb) {
    Scene* s = (Scene*)sp;
    Vec3 cx, cy;
    camera_basis(*s, width, height, cx, cy);
    int num_samples = spp / 4;
    for (long i = 0; i < n; ++i) {
        Sampler sm;
        sm.pixel = (uint32_t)(py_img[i] * width + px[i]);
        sm.sample = (uint32_t)sample_idx[i];
        sm.k0 = (uint32_t)seed; sm.k1 = (uint32_t)(seed >> 32);
        int subi = sample_idx[i] / num_samples;
        int sy = subi / 2, sx = subi % 2;
        double u[4];
        sm.block(0, 0, u);
        Ray r = camera_ray(*s, cx, cy, px[i], height - py_img[i] - 1, width, height, sx, sy, tent(u[0]), tent(u[1]));
        Vec3 L = s->received_radiance(r, sm, nullptr);
        rgb[3 * i] = L.x; rgb[3 * i + 1] = L.y; rgb[3 * i + 2] = L.z;
    }
}

void or_philox(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1, uint32_t* out4) {
    Philox::gen(c0, c1, c2, c3, k0, k1, out4);
}

}  // extern "C"
