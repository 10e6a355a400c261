"""The f64 oracle with rough metal (brdf 4, GGX microfacet reflection, DESIGN §3g), for the metal tests.

It starts from lights_oracle.source() (the glass oracle plus estimator 3) and adds the metal branch the same way: each
addition below is inserted at an anchor that must occur exactly once, so a change of the anchor's code fails loudly instead of
building something else.  Every other material and estimator of the copy runs exactly the code it ran before.  The TOML variant
`type = "metal"` is added to glass_oracle's parsing.  The library is compiled once per process into a temporary directory (the
tree stays read-only) and driven through glass_oracle's OracleScene.
"""
import ctypes as C
import math
import os
import subprocess
import tempfile
import threading

import numpy as np

import glass_oracle as G
import lights_oracle as LO
from oracle import oracle as O

ACCEL_OCTREE_FAITHFUL, ACCEL_EXACT, EST_NEE, EST_NEE_ALL_LIGHTS = G.ACCEL_OCTREE_FAITHFUL, G.ACCEL_EXACT, G.EST_NEE, LO.EST_NEE_ALL_LIGHTS
MIN_ROUGHNESS = 0.05

# (anchor, text inserted right after it)
ADDITIONS = [
    ("""enum BrdfKind { B_DIFFUSE = 0, B_SPECULAR = 1, B_PHONG = 2, B_DIELECTRIC = 3 };
""", """constexpr int B_METAL = 4;  // rough metal: k = {roughness, alpha = roughness^2, 0}, color_s = F0
"""),
    # or_add_object: params {roughness, F0[3]}
    ("""    o.r = 0; o.pos = V(0, 0, 0); o.n = V(0, 0, 0);
""", """    if (brdf_kind == B_METAL) {
        o.brdf.k = V(bp[0], bp[0] * bp[0], 0);
        o.brdf.color_s = V(bp[1], bp[2], bp[3]);
    }
"""),
    # f of rule 4, for every light sample that evaluates the material (estimator 3's included)
    ("""            case B_DIFFUSE: return f.k * FRAC_1_PI;
""", """            case B_METAL: return metal_f(f, n, o, i);
"""),
    # the GGX rules, stated directly
    ("""    // ---- create_local_coord  src/scene.rs:112-123
""", r"""    // ---- rough metal (DESIGN §3g): D, Smith's Lambda, Schlick's F, f = F D G2 / (4 (n.o)(n.i)), Heitz 2018's visible normals
    static double metal_lambda(double a2, double c) { return (std::sqrt(1. + a2 * (1. - c * c) / (c * c)) - 1.) / 2.; }
    static Vec3 metal_F(const BRDF& f, double oh) {
        const double m = 1. - oh, m5 = m * m * m * m * m;
        return f.color_s + (V(1, 1, 1) - f.color_s) * m5;
    }
    static Vec3 metal_f(const BRDF& f, const Vec3& n, const Vec3& o, const Vec3& i) {
        const double no = dot(n, o), ni = dot(n, i);
        if (no <= 0. || ni <= 0.) return V(0, 0, 0);
        const double a2 = f.k.y * f.k.y;
        const Vec3 h = norm(o + i);
        const double nh = dot(n, h), q = nh * nh * (a2 - 1.) + 1.;
        const double D = a2 / (PI * q * q);
        const double G2 = 1. / (1. + metal_lambda(a2, no) + metal_lambda(a2, ni));
        return metal_F(f, dot(o, h)) * (D * G2 / (4. * no * ni));
    }
    // the continuation: i and its weight F G2 / G1(o); false = the path ends (n.i <= 0)
    static bool metal_sample(const BRDF& f, const Vec3& n, const Vec3& o, double u1, double u2, Vec3& i, Vec3& w) {
        Vec3 tu, tv, tw;
        create_local_coord(n, tu, tv, tw);
        const double alpha = f.k.y, oz = dot(o, n);
        const Vec3 vh = norm(V(alpha * dot(o, tu), alpha * dot(o, tv), oz));
        const double lensq = vh.x * vh.x + vh.y * vh.y;
        const Vec3 t1 = lensq > 0. ? V(-vh.y, vh.x, 0) * (1. / std::sqrt(lensq)) : V(1, 0, 0);
        const Vec3 t2 = cross(vh, t1);
        const double r = std::sqrt(u1), phi = 2. * PI * u2;
        const double p1 = r * std::cos(phi), s = 0.5 * (1. + vh.z);
        const double p2 = (1. - s) * std::sqrt(std::max(1. - p1 * p1, 0.)) + s * r * std::sin(phi);
        const Vec3 nh = t1 * p1 + t2 * p2 + vh * std::sqrt(std::max(0., 1. - p1 * p1 - p2 * p2));
        const Vec3 ne = norm(V(alpha * nh.x, alpha * nh.y, std::max(0., nh.z)));
        const Vec3 h = tu * ne.x + tv * ne.y + n * ne.z;
        const double oh = dot(o, h);
        i = h * (2. * oh) - o;
        const double ni = dot(n, i);
        if (oz <= 0. || ni <= 0.) return false;
        const double a2 = alpha * alpha, lo = metal_lambda(a2, oz);
        w = metal_F(f, oh) * ((1. + lo) / (1. + lo + metal_lambda(a2, ni)));
        return true;
    }

"""),
    # the metal vertex, after the dielectric's: a diffuse vertex's light sample with f of rule 4 and the TRUE o, roulette as
    # for a diffuse vertex, one visible-normal continuation
    ("""                    rad = mult(objects[h2.id].emitted + reflected_radiance(h2, -i, depth + 1, s, cnt), w) / p;
            }
            return rad;
        }
""", """        if (obj.brdf.kind == B_METAL) {
            const Vec3 om = -hit.dir;  // never the stale `o` a mirror in front hands the recursion
            Vec3 rad = V(0, 0, 0);
            if (estimator == 3) {
                rad = all_lights_direct(obj, x, n, om, b0, sel, cnt);
            } else {
                Vec3 y, ny;
                double pdf;
                light_sample(b0, y, ny, pdf);
                Vec3 i = norm(y - x);
                double r_sqr = dot(y - x, y - x);
                double visibility = mutually_visible(x, y, cnt) ? 1. : 0.;
                rad = mult(objects[light_source].emitted, metal_f(obj.brdf, n, om, i)) * visibility * dot(n, i) *
                      dot(ny, -i) / (r_sqr * pdf);
            }
            if (b0[2] < p) {
                Vec3 i, w;
                if (metal_sample(obj.brdf, n, om, b1[0], b1[1], i, w)) {
                    Hit h2{};
                    if (trace_ray(Ray{x, i}, h2, cnt)) {
                        if (estimator == 3 && light_of[(size_t)h2.id] < 0)   // not sampled by the light sample
                            rad += mult(objects[h2.id].emitted, w) / p;
                        rad += mult(reflected_radiance(h2, -i, depth + 1, s, cnt), w) / p;
                    }
                }
            }
            return rad;
        }
"""),
]


def source() -> str:
    src = LO.source()
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
            d = tempfile.mkdtemp(prefix="metal_oracle_")
            with open(os.path.join(d, "metal_oracle.cpp"), "w") as f:
                f.write(source())
            out = os.path.join(d, "libmetal_oracle.so")
            subprocess.run(["/usr/bin/g++", *G.CXXFLAGS, "-o", out, os.path.join(d, "metal_oracle.cpp")], check=True, capture_output=True)
            L, ref = C.CDLL(out), O.lib()
            for name in dir(ref):   # the same entry points as the oracle's, with the same signatures
                if name.startswith("or_"):
                    f, g = getattr(L, name), getattr(ref, name)
                    f.argtypes, f.restype = g.argtypes, g.restype
            _lib = L
    return _lib


def brdf(b, vec):
    """glass_oracle._brdf plus `type = "metal"`: (4, [roughness, F0 r, g, b]) with the loader's checks"""
    if b["type"] != "metal":
        return _glass_brdf(b, vec)
    rough = b["roughness"]
    if isinstance(rough, bool) or not isinstance(rough, (int, float)) or not (math.isfinite(rough) and MIN_ROUGHNESS <= rough <= 1):
        raise O.OracleError("parse: metal roughness must be finite and in [0.05, 1]")
    color = list(map(float, b.get("color", [1.0, 1.0, 1.0])))
    if len(color) != 3 or not all(0.0 <= c <= 1.0 for c in color):
        raise O.OracleError("parse: metal color must be 3 numbers in [0, 1]")
    return 4, np.array([float(rough)] + color)


_glass_brdf = G._brdf


class OracleScene(G.OracleScene):
    """glass_oracle.OracleScene on the oracle with metal (and estimator 3)"""

    _mu = threading.Lock()

    def __init__(self, spec: dict, assets_dir: str | None = None):
        # glass_oracle.OracleScene builds its scene through glass_oracle.lib() and glass_oracle._brdf: for the duration of one
        # construction those name this module's library and parser (one construction at a time)
        with OracleScene._mu:
            old = G.lib, G._brdf
            G.lib, G._brdf = lib, brdf
            try:
                super().__init__(spec, assets_dir)
            finally:
                G.lib, G._brdf = old
