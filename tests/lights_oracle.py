"""The f64 glass oracle (tests/glass_oracle.cpp) with estimator 3, next-event estimation over every emitting sphere and mesh
(RTB_EST_NEE_ALL_LIGHTS, DESIGN §3f), for the all-lights tests.

glass_oracle.cpp stays the reference of the glass tests as it is.  This module adds estimator 3 to a copy of its source at
compile time: each addition below is inserted at an anchor that must occur exactly once, so a change of the anchor's code
fails loudly instead of building something else.  Estimators 0 and 1 of the copy run exactly the original code.  The library is
compiled once per process into a temporary directory (the tree stays read-only) and driven through glass_oracle's OracleScene.
"""
import ctypes as C
import os
import subprocess
import tempfile
import threading

import glass_oracle as G
from oracle import oracle as O

EST_NEE_ALL_LIGHTS = 3
ACCEL_OCTREE_FAITHFUL, ACCEL_EXACT = G.ACCEL_OCTREE_FAITHFUL, G.ACCEL_EXACT

# (anchor, text inserted right after it)
ADDITIONS = [
    # the light table, built once the objects are final
    ("""    int estimator = 0;  // 0 NEE live, 1 dead MIS branch
    std::string err;
""", r"""    // estimator 3: the light table (object, probability, area, triangle cdf of a mesh), and each object's entry or -1
    struct LightEntry {
        long obj;
        double prob, area;
        std::vector<double> tri_cdf;
    };
    std::vector<LightEntry> lights;
    std::vector<double> light_cdf;
    std::vector<long> light_of;

    // weight lum709(max(emitted, 0)) * area of every sphere and mesh, in object order; planes and zero weights stay out
    void build_lights() {
        lights.clear();
        light_cdf.clear();
        light_of.assign(objects.size(), -1);
        double total = 0.;
        for (size_t k = 0; k < objects.size(); ++k) {
            const Object& ob = objects[k];
            if (ob.gkind == G_PLANE) continue;
            const Vec3& e = ob.emitted;
            const double lum = 0.2126 * std::max(e.x, 0.) + 0.7152 * std::max(e.y, 0.) + 0.0722 * std::max(e.z, 0.);
            LightEntry L{(long)k, 0., 0., {}};
            if (ob.gkind == G_SPHERE) L.area = 4. * PI * ob.r * ob.r;
            else {
                for (size_t t = 0; t < ob.mesh.num_triangles(); ++t) {
                    const Triangle tr = ob.mesh.triangle(t);
                    L.area += 0.5 * mag(cross(tr.b - tr.a, tr.c - tr.a));
                    L.tri_cdf.push_back(L.area);
                }
                for (double& c : L.tri_cdf) c /= L.area;
            }
            const double w = lum * L.area;
            if (!(w > 0.)) continue;
            L.prob = w;
            total += w;
            light_of[k] = (long)lights.size();
            lights.push_back(L);
        }
        double cum = 0.;
        for (LightEntry& L : lights) {
            L.prob /= total;
            cum += L.prob;
            light_cdf.push_back(cum);
        }
    }
    // partition_point(cdf <= u), clamped to the last entry
    static size_t pick(const std::vector<double>& cdf, double u) {
        const size_t i = std::upper_bound(cdf.begin(), cdf.end(), u) - cdf.begin();
        return i < cdf.size() ? i : cdf.size() - 1;
    }
    // estimator 3's light sample at x: one light of the table by power, one point of it; clamped cosines, two-sided emitters
    Vec3 all_lights_direct(const Object& obj, const Vec3& x, const Vec3& n, const Vec3& o, const double b0[4], const double sel[4],
                           Counters* cnt) const {
        if (lights.empty()) return V(0, 0, 0);
        const LightEntry& L = lights[pick(light_cdf, sel[2])];
        const Object& lo = objects[(size_t)L.obj];
        Vec3 y, ny;
        if (lo.gkind == G_SPHERE) {  // the reference's sphere sampler
            const double z = 2. * b0[0] - 1.;
            Vec3 d = norm(V(std::sqrt(1.0 - z * z) * std::cos(2. * PI * b0[1]), std::sqrt(1.0 - z * z) * std::sin(2. * PI * b0[1]), z));
            y = lo.pos + d * lo.r;
            ny = d;
        } else {  // a triangle by true area, a uniform point of it
            const Triangle t = lo.mesh.triangle(pick(L.tri_cdf, sel[1]));
            const double sq = std::sqrt(b0[0]);
            y = t.a * (1. - sq) + t.b * (sq * (1. - b0[1])) + t.c * (sq * b0[1]);
            ny = t.normal();
        }
        const Vec3 i = norm(y - x);
        const double g = std::max(dot(n, i), 0.) * std::fabs(dot(ny, -i)) / (dot(y - x, y - x) * (L.prob / L.area));
        if (g > 0. && mutually_visible(x, y, cnt)) return mult(lo.emitted, brdf_eval(obj.brdf, n, o, i)) * g;
        return V(0, 0, 0);
    }
"""),
    # the light sample: estimator 3 replaces the live-NEE branch
    ("""            rad = rad_direct;
        }""", """ else if (estimator == 3) {
            rad = all_lights_direct(obj, x, n, o, b0, sel, cnt);
        }"""),
    # the continuation: emission of an emitter outside the table counts where the path meets it
    ("""            brdf_sample(obj.brdf, n, o, b1, i, pdf_brdf);
            Hit h2{};
            if (trace_ray(Ray{x, i}, h2, cnt)) {
""", """                if (estimator == 3 && light_of[(size_t)h2.id] < 0)   // not sampled by the light sample
                    rad += mult(objects[h2.id].emitted, brdf_eval(obj.brdf, n, o, i)) * dot(n, i) / (pdf_brdf * p);
"""),
    ("""        if (!equal_within(s->objects[i].emitted, V(0, 0, 0), 0.00001)) { s->light_source = (long)i; break; }
""", """    s->build_lights();
"""),
]


def source() -> str:
    src = open(G.SRC).read()
    for anchor, text in ADDITIONS:
        assert src.count(anchor) == 1, anchor
        src = src.replace(anchor, anchor + text)
    return src


_lib = None
_mu = threading.Lock()


def lib():
    global _lib
    with _mu:
        if _lib is None:
            d = tempfile.mkdtemp(prefix="lights_oracle_")
            with open(os.path.join(d, "lights_oracle.cpp"), "w") as f:
                f.write(source())
            out = os.path.join(d, "liblights_oracle.so")
            subprocess.run(["/usr/bin/g++", *G.CXXFLAGS, "-o", out, os.path.join(d, "lights_oracle.cpp")], check=True, capture_output=True)
            L, ref = C.CDLL(out), O.lib()
            for name in dir(ref):   # the same entry points as the oracle's, with the same signatures
                if name.startswith("or_"):
                    f, g = getattr(L, name), getattr(ref, name)
                    f.argtypes, f.restype = g.argtypes, g.restype
            _lib = L
    return _lib


class OracleScene(G.OracleScene):
    """glass_oracle.OracleScene on the oracle with estimator 3"""

    def __init__(self, spec: dict, assets_dir: str | None = None):
        with _swap_lib():
            super().__init__(spec, assets_dir)


class _swap_lib:
    """glass_oracle.OracleScene builds its scene through glass_oracle.lib(): for the duration of one construction that names
    this module's library instead (one construction at a time)"""

    _mu = threading.Lock()

    def __enter__(self):
        self._mu.acquire()
        self._old = G.lib
        G.lib = lib

    def __exit__(self, *exc):
        G.lib = self._old
        self._mu.release()
