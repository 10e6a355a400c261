"""Rough metal (brdf 4) without a GPU: the GGX header (csrc/microfacet_rule.cuh) against a numpy f64 restatement of D, G1, G2
and Schlick, its sampler against its pdf (quadrature and a chi-square test), reciprocity and energy, and the loader on
host-only handles."""
import os
import subprocess

import numpy as np
import pytest
from scipy import stats
from scipy.special import roots_legendre

from conftest import ROOT

NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
ALPHAS = [0.0025, 0.04, 0.25, 1.0]
COS_O = [0.1, 0.5, 0.99]

CAMERA = """
[camera]
pos = [0.0, 0.0, 10.0]
dir = [0.0, 0.0, -1.0]
"""
LIGHT = """
[[objects]]
emitted = [4.0, 4.0, 4.0]
brdf = { type = "diffuse", kd = [0.0, 0.0, 0.0] }
geometry = { type = "sphere", pos = [0.0, 5.0, 0.0], r = 1.0 }
"""


def scene(brdf):
    return CAMERA + LIGHT + f"""
[[objects]]
brdf = {brdf}
geometry = {{ type = "sphere", pos = [0.0, 0.0, 0.0], r = 1.0 }}
"""


def load(rtb, text):
    return rtb.Scene.from_toml_string(text, device=-1)


# ---- loader --------------------------------------------------------------------------------------------------------------
def test_toml_fields(rtb):
    o = load(rtb, scene('{ type = "metal", roughness = 0.3, color = [1.0, 0.71, 0.29] }')).object(1)
    assert o["brdf"] == 4 and o["k"] == pytest.approx([0.3, 0.09, 0.0], rel=1e-15) and o["color_s"] == [1.0, 0.71, 0.29]
    o = load(rtb, scene('{ type = "metal", roughness = 1 }')).object(1)       # an integer is a number; color defaults to 1
    assert o["k"] == [1.0, 1.0, 0.0] and o["color_s"] == [1.0, 1.0, 1.0]
    assert load(rtb, scene('{ type = "metal", roughness = 0.05 }')).object(1)["k"][0] == 0.05


@pytest.mark.parametrize("brdf, field", [
    ('{ type = "metal" }', "roughness"),
    ('{ type = "metal", roughness = 0.0 }', "roughness"),
    ('{ type = "metal", roughness = 0.049 }', "roughness"),
    ('{ type = "metal", roughness = 1.01 }', "roughness"),
    ('{ type = "metal", roughness = inf }', "roughness"),
    ('{ type = "metal", roughness = nan }', "roughness"),
    ('{ type = "metal", roughness = "rough" }', "roughness"),
    ('{ type = "metal", roughness = 0.3, color = [1.0, 1.5, 1.0] }', "color"),
    ('{ type = "metal", roughness = 0.3, color = [-0.1, 1.0, 1.0] }', "color"),
    ('{ type = "metal", roughness = 0.3, color = [1.0, 1.0] }', "color"),
    ('{ type = "metal", roughness = 0.3, color = "gold" }', "color"),
])
def test_invalid_fields_name_the_field(rtb, brdf, field):
    with pytest.raises(rtb.LoadTomlError) as e:
        load(rtb, scene(brdf))
    assert e.value.code == rtb.RTB_EPARSE and field in str(e.value)


def test_unknown_variant_lists_metal(rtb):
    with pytest.raises(rtb.LoadTomlError) as e:
        load(rtb, scene('{ type = "gold", roughness = 0.3 }'))
    assert e.value.code == rtb.RTB_EPARSE and "`metal`" in str(e.value) and "`dielectric`" in str(e.value)


def _objects(brdf):
    return [
        {"emitted": (4.0, 4.0, 4.0), "brdf": ("diffuse", (0.0, 0.0, 0.0)), "geometry": ("sphere", (0.0, 5.0, 0.0), 1.0)},
        {"brdf": brdf, "geometry": ("sphere", (0.0, 0.0, 0.0), 1.0)},
    ]


def test_scene_create_and_object_round_trip(rtb):
    sc = rtb.Scene.from_objects((0, 0, 10), (0, 0, -1), _objects(("metal", 0.3, (0.95, 0.64, 0.54))), device=-1)
    o = sc.object(1)
    assert o["brdf"] == 4 and o["k"] == pytest.approx([0.3, 0.09, 0.0], rel=1e-15) and o["color_s"] == [0.95, 0.64, 0.54]
    # what rtb_scene_object reports builds the same object again
    again = rtb.Scene.from_objects((0, 0, 10), (0, 0, -1), _objects(("metal", o["k"][0], o["color_s"])), device=-1).object(1)
    assert again == o
    assert rtb.Scene.from_objects((0, 0, 10), (0, 0, -1), _objects(("metal", 0.5)), device=-1).object(1)["color_s"] == [1.0, 1.0, 1.0]
    for bad in (("metal", 0.01), ("metal", 1.5), ("metal", float("nan")), ("metal", 0.3, (1.0, 2.0, 1.0)), ("metal", 0.3, (0.5, -0.5, 1.0))):
        with pytest.raises(rtb.LoadTomlError) as e:
            rtb.Scene.from_objects((0, 0, 10), (0, 0, -1), _objects(bad), device=-1)
        assert e.value.code == rtb.RTB_EPARSE and "metal" in str(e.value)


def test_export_import_round_trip(rtb):
    sc = load(rtb, scene('{ type = "metal", roughness = 0.08, color = [0.91, 0.92, 0.92] }'))
    again = rtb.Scene.from_export(sc.export(), device=-1)
    assert [again.object(i) for i in range(2)] == [sc.object(i) for i in range(2)]
    assert again.object(1)["brdf"] == 4


# ---- numpy f64 restatement of the rule (DESIGN §3g) ------------------------------------------------------------------------
def _dot(a, b):
    return np.einsum("...j,...j->...", a, b)


def D_np(a2, nh):
    q = nh * nh * (a2 - 1) + 1
    return a2 / (np.pi * q * q)


def lambda_np(a2, c):
    return (np.sqrt(1 + a2 * (1 - c * c) / (c * c)) - 1) / 2


def G1_np(a2, c):
    return 1 / (1 + lambda_np(a2, c))


def G2_np(a2, co, ci):
    return 1 / (1 + lambda_np(a2, co) + lambda_np(a2, ci))


def schlick_np(F0, oh):
    return F0 + (1 - F0) * (1 - oh)[..., None] ** 5


def half(o, i):
    h = o + i
    return h / np.linalg.norm(h, axis=-1, keepdims=True)


def _unit(v):
    return v / np.linalg.norm(v, axis=-1, keepdims=True)


# The restatement takes n, o and i as the unit vectors the rule is stated for.  The fp32 inputs of the header are unit only to
# within an ulp; a polished lobe (alpha^2 = 6e-6) is narrow enough for that ulp to matter in the literal denominator of D, which
# is why the header writes it as sin^2 + alpha^2 cos^2 (microfacet_rule.cuh).
def f_np(F0, alpha, n, o, i):
    """f(o, i) = F D G2 / (4 (n.o)(n.i)), 0 unless both lie above"""
    n, o, i = _unit(n), _unit(o), _unit(i)
    a2, no, ni = alpha * alpha, _dot(n, o), _dot(n, i)
    h = half(o, i)
    with np.errstate(all="ignore"):
        v = schlick_np(F0, _dot(o, h)) * (D_np(a2, _dot(n, h)) * G2_np(a2, no, ni) / (4 * no * ni))[..., None]
    return np.where(((no > 0) & (ni > 0))[..., None], v, 0.0)


def pdf_np(alpha, n, o, i, clamp=True):
    """G1(o) D(h) / (4 n.o) (D is 0 for microfacet normals with n.h <= 0); clamp: 0 where n.i <= 0 (the path ends there)"""
    n, o, i = _unit(n), _unit(o), _unit(i)
    a2, no, h = alpha * alpha, _dot(n, o), half(o, i)
    with np.errstate(all="ignore"):
        v = np.where(_dot(n, h) > 0, G1_np(a2, no) * D_np(a2, _dot(n, h)) / (4 * no), 0.0)
    return np.where(_dot(n, i) > 0, v, 0.0) if clamp else v


# ---- the header through a host harness -------------------------------------------------------------------------------------
HARNESS = r"""
#include <cstdio>
#include "microfacet_rule.cuh"
using namespace rtb;
// stdin: mode, n, then n records of 14 floats; stdout: n records of 11 floats
//   mode 0 (sample): {n, o, alpha, F0, u1, u2, -}  -> {i, ok, w, f(o, i), pdf(o, i)}
//   mode 1 (eval):   {n, o, i, alpha, F0, -}       -> {f(o, i), pdf(o, i), f(i, o), -...}
int main() {
    int mode, n;
    if (fread(&mode, 4, 1, stdin) != 1 || fread(&n, 4, 1, stdin) != 1) return 1;
    for (int k = 0; k < n; ++k) {
        float r[14];
        if (fread(r, 4, 14, stdin) != 14) return 1;
        const float3 nn = make_float3(r[0], r[1], r[2]), o = make_float3(r[3], r[4], r[5]);
        float out[11] = {0};
        if (mode == 0) {
            const float3 F0 = make_float3(r[7], r[8], r[9]);
            float3 i = make_float3(0, 0, 0), w = make_float3(0, 0, 0);
            const bool ok = metal_sample(F0, r[6], nn, o, r[10], r[11], i, w);
            const float3 f = metal_eval(F0, r[6], nn, o, i);
            const float o11[11] = {i.x, i.y, i.z, ok ? 1.0f : 0.0f, w.x, w.y, w.z, f.x, f.y, f.z, metal_pdf(r[6], nn, o, i)};
            for (int j = 0; j < 11; ++j) out[j] = o11[j];
        } else {
            const float3 i = make_float3(r[6], r[7], r[8]), F0 = make_float3(r[10], r[11], r[12]);
            const float3 f = metal_eval(F0, r[9], nn, o, i), g = metal_eval(F0, r[9], nn, i, o);
            const float o7[7] = {f.x, f.y, f.z, metal_pdf(r[9], nn, o, i), g.x, g.y, g.z};
            for (int j = 0; j < 7; ++j) out[j] = o7[j];
        }
        fwrite(out, 4, 11, stdout);
    }
    return 0;
}
"""


@pytest.fixture(scope="module")
def rule(tmp_path_factory):
    d = tmp_path_factory.mktemp("microfacet_rule")
    (d / "h.cu").write_text(HARNESS)
    exe = d / "h"
    subprocess.run([NVCC, "-std=c++17", "-O2", "-ccbin", "/usr/bin/g++", "-I", os.path.join(ROOT, "raytracer-server_b200", "csrc"),
                    str(d / "h.cu"), "-o", str(exe)], check=True)

    def run(mode, rec):
        rec = np.ascontiguousarray(np.pad(rec, ((0, 0), (0, 14 - rec.shape[1]))), dtype=np.float32)
        inp = np.int32(mode).tobytes() + np.int32(len(rec)).tobytes() + rec.tobytes()
        out = subprocess.run([str(exe)], input=inp, capture_output=True, check=True).stdout
        return np.frombuffer(out, np.float32).reshape(len(rec), 11).astype(np.float64)

    def sample(n, o, alpha, F0, u):
        m = len(u)
        rec = np.concatenate([np.broadcast_to(n, (m, 3)), np.broadcast_to(o, (m, 3)), np.full((m, 1), alpha),
                              np.broadcast_to(F0, (m, 3)), u], 1)
        r = run(0, rec)
        return {"i": r[:, :3], "ok": r[:, 3] == 1, "w": r[:, 4:7], "f": r[:, 7:10], "pdf": r[:, 10]}

    def evaluate(n, o, i, alpha, F0):
        m = len(i)
        rec = np.concatenate([np.broadcast_to(n, (m, 3)), np.broadcast_to(o, (m, 3)), i, np.broadcast_to(np.reshape(alpha, (-1, 1)), (m, 1)),
                              np.broadcast_to(F0, (m, 3))], 1)
        r = run(1, rec)
        return {"f": r[:, :3], "pdf": r[:, 3], "f_swapped": r[:, 4:7]}

    return {"sample": sample, "eval": evaluate}


def _f32(x):
    return np.asarray(x, np.float64).astype(np.float32).astype(np.float64)


def _case(cos_o, tilt=0.3):
    """a unit normal away from the axes (so that the frame is a generic one) and o at n.o = cos_o, both exact in fp32"""
    n = np.array([np.sin(tilt) * 0.6, np.sin(tilt) * 0.8, np.cos(tilt)])
    u = np.cross([0.0, 1.0, 0.0], n)
    u /= np.linalg.norm(u)
    o = cos_o * n + np.sqrt(1 - cos_o ** 2) * u
    n, o = _f32(n), _f32(o)
    return n, o


def _around(n, o):
    """the mirror direction r of o about n and an orthonormal pair around it"""
    n, o = _unit(n), _unit(o)
    r = 2 * _dot(o, n) * n - o
    e1 = np.cross(r, n if abs(_dot(r, n)) < 0.9 else [1.0, 0.0, 0.0])
    e1 /= np.linalg.norm(e1)
    return r, e1, np.cross(r, e1)


def _psi_edges(alpha, top=np.pi):
    e = [0.0] + [alpha * 2.0 ** k for k in range(-3, 12) if alpha * 2.0 ** k < top] + [top]
    return np.array(e)


def _grid(n, o, alpha, n_chi=2048, n_gl=48):
    """quadrature nodes over the directions i, placed through their half vectors h: polar coordinates (psi, chi) of h around n,
    Gauss-Legendre in psi, piecewise on a scale of alpha (the width of D), and the periodic trapezoid rule in chi; i = 2 (o.h) h
    - o with d(omega_i) = 4 (o.h) d(omega_h) over the h with o.h > 0.  Returns (directions i, weights)."""
    nu = _unit(n)
    e1 = _unit(np.cross(nu, [1.0, 0.0, 0.0]))
    e2 = np.cross(nu, e1)
    x, wx = roots_legendre(n_gl)
    edges = _psi_edges(alpha, np.pi / 2)    # D is 0 beyond the horizon of n
    psi = np.concatenate([(a + b) / 2 + (b - a) / 2 * x for a, b in zip(edges[:-1], edges[1:])])
    wpsi = np.concatenate([(b - a) / 2 * wx for a, b in zip(edges[:-1], edges[1:])]) * np.sin(psi)
    chi = np.arange(n_chi) * (2 * np.pi / n_chi)
    P, X = np.meshgrid(psi, chi, indexing="ij")
    h = (np.cos(P)[..., None] * nu + np.sin(P)[..., None] * (np.cos(X)[..., None] * e1 + np.sin(X)[..., None] * e2)).reshape(-1, 3)
    oh = _dot(h, _unit(o))
    w = np.broadcast_to(wpsi[:, None] * (2 * np.pi / n_chi), P.shape).reshape(-1) * 4 * oh
    keep = oh > 0
    return (2 * oh[keep, None] * h[keep] - _unit(o)), w[keep]


@pytest.mark.parametrize("alpha", ALPHAS)
@pytest.mark.parametrize("cos_o", COS_O)
def test_pdf_integrates_to_one(rule, alpha, cos_o):
    n, o = _case(cos_o)
    d, w = _grid(n, o, alpha)
    # the unclamped pdf over the whole sphere: the visible normals are a distribution
    whole = (pdf_np(alpha, n, o, d, clamp=False) * w).sum()
    assert abs(whole - 1) < 1e-3, whole
    # the header's pdf over the upper hemisphere + the mass that reflects below the horizon (where the path ends) = 1
    upper = (rule["eval"](n, o, d, alpha, np.ones(3))["pdf"] * w).sum()
    below = (np.where(_dot(d, n) <= 0, pdf_np(alpha, n, o, d, clamp=False), 0.0) * w).sum()
    assert abs(upper + below - 1) < 2e-3, (upper, below)
    if alpha == ALPHAS[0] and cos_o >= 0.5:     # a polished lobe well above the horizon: only GGX's O(alpha^2) tail is lost
        assert abs(upper - 1) < 1e-4 and below < 1e-4


@pytest.mark.parametrize("alpha", ALPHAS)
@pytest.mark.parametrize("cos_o", COS_O)
def test_samples_follow_the_pdf(rule, alpha, cos_o):
    n, o = _case(cos_o)
    m = 100_000
    F0 = np.array([1.0, 0.71, 0.29])
    u = np.random.default_rng(int(alpha * 1e4) + int(cos_o * 100)).random((m, 2))
    s = rule["sample"](n, o, alpha, F0, u)
    ok, i = s["ok"], s["i"]
    assert np.abs(np.linalg.norm(i, axis=1) - 1).max() < 1e-5
    assert (_dot(i[ok], n) > 0).all() and (_dot(i[~ok], n) <= 1e-6).all()
    # chi-square on a grid of (psi, chi) cells around the mirror direction, plus one cell for the paths that end
    r, e1, e2 = _around(n, o)
    edges = _psi_edges(alpha)
    n_chi = 8

    def cells(d):   # psi from atan2: arccos loses the small angles of a polished lobe
        psi = np.arctan2(np.linalg.norm(np.cross(d, r), axis=1), _dot(d, r))
        chi = np.mod(np.arctan2(_dot(d, e2), _dot(d, e1)), 2 * np.pi)
        return np.clip(np.searchsorted(edges, psi, side="right") - 1, 0, len(edges) - 2) * n_chi + np.minimum((chi / (2 * np.pi) * n_chi).astype(int), n_chi - 1)

    cell = np.where(ok, cells(i), (len(edges) - 1) * n_chi)
    obs = np.bincount(cell, minlength=(len(edges) - 1) * n_chi + 1).astype(float)
    d, w = _grid(n, o, alpha)
    dcell = cells(d)
    p_all = pdf_np(alpha, n, o, d, clamp=False) * w
    up = _dot(d, n) > 0
    exp = np.bincount(dcell[up], weights=p_all[up], minlength=len(obs))
    exp[-1] = p_all[~up].sum()
    exp *= m / exp.sum()
    big = exp >= 20
    o_, e_ = np.append(obs[big], obs[~big].sum()), np.append(exp[big], exp[~big].sum())
    keep = e_ > 0
    chi2, pv = stats.chisquare(o_[keep], e_[keep] * o_[keep].sum() / e_[keep].sum())
    assert big.sum() >= 10 and pv > 1e-4, (chi2, pv, big.sum())     # twelve cases: a false alarm in about 0.1 % of runs
    # the weight of every sample is f (n.i) / pdf of rules 4 and 5, F(o.h) G2 / G1(o)
    ni = _dot(n, i[ok])
    want = f_np(F0, alpha, n, o, i[ok]) * (ni / pdf_np(alpha, n, o, i[ok]))[:, None]
    good = ni > 1e-3        # fp32 n.i of an almost grazing sample carries a large relative error of its own
    assert good.mean() > 0.5
    rel = np.abs(s["w"][ok][good] / want[good] - 1)
    assert rel.max() < 1e-4, rel.max()
    assert np.abs(s["w"][ok] / want - 1).max() < 1e-2
    # and it is what the header's own f and pdf give
    assert np.abs(s["w"][ok][good] / (s["f"][ok][good] * (ni[good] / s["pdf"][ok][good])[:, None]) - 1).max() < 1e-4


def test_eval_against_numpy_and_reciprocity(rule):
    rng = np.random.default_rng(7)
    m = 20000
    n = rng.normal(size=(m, 3))
    n /= np.linalg.norm(n, axis=1, keepdims=True)
    o, i = rng.normal(size=(m, 3)), rng.normal(size=(m, 3))
    o *= np.sign(_dot(o, n))[:, None]
    i *= np.sign(_dot(i, n))[:, None]
    o /= np.linalg.norm(o, axis=1, keepdims=True)
    i /= np.linalg.norm(i, axis=1, keepdims=True)
    # half of the pairs near the specular peak, where the lobe of a polished metal lives
    r = 2 * _dot(o, n)[:, None] * n - o
    near = np.arange(m) < m // 2
    i[near] = r[near] + 0.01 * rng.normal(size=(near.sum(), 3))
    i /= np.linalg.norm(i, axis=1, keepdims=True)
    n, o, i = _f32(n), _f32(o), _f32(i)
    alpha = _f32(rng.choice(ALPHAS + [0.09, 0.6], m))
    F0 = _f32(rng.random((m, 3)))
    keep = (_dot(n, o) > 0.02) & (_dot(n, i) > 0.02)
    n, o, i, alpha, F0 = n[keep], o[keep], i[keep], alpha[keep], F0[keep]
    e = rule["eval"](n, o, i, alpha, F0)
    f = f_np(F0, alpha, n, o, i)
    pdf = pdf_np(alpha, n, o, i)
    assert np.abs(e["f"] / f - 1).max() < 3e-4
    assert np.abs(e["pdf"] / pdf - 1).max() < 3e-4
    assert np.abs(e["f_swapped"] / e["f"] - 1).max() < 3e-5          # f(o, i) = f(i, o), to fp32 rounding
    # the pieces: D at the peak, G1 and G2 at normal incidence, Schlick's end points
    assert D_np(0.01, np.array(1.0)) == pytest.approx(1 / (np.pi * 0.01))
    assert G1_np(0.3, np.array(1.0)) == 1 and G2_np(0.3, np.array(1.0), np.array(1.0)) == 1
    assert np.allclose(schlick_np(np.array([0.2, 0.5, 1.0]), np.array(1.0)), [0.2, 0.5, 1.0])
    assert np.allclose(schlick_np(np.array([0.2, 0.5, 1.0]), np.array(0.0)), 1.0)
    # below the horizon on either side: 0
    z = rule["eval"](n[:10], o[:10], -i[:10], alpha[:10], F0[:10])
    assert (z["f"] == 0).all() and (z["pdf"] == 0).all()


def test_albedo_is_at_most_one(rule):
    albedo = {}
    for cos_o in COS_O:
        n, o = _case(cos_o)
        for alpha in ALPHAS:
            d, w = _grid(n, o, alpha)
            quad = (f_np(np.ones(3), alpha, n, o, d)[:, 0] * np.clip(_dot(d, n), 0, None) * w).sum()
            u = np.random.default_rng(3).random((50_000, 2))
            s = rule["sample"](n, o, alpha, np.ones(3), u)
            mc = np.where(s["ok"], s["w"][:, 0], 0.0).mean()
            assert quad <= 1 + 1e-3 and mc <= 1, (cos_o, alpha, quad, mc)
            assert abs(mc - quad) < 0.01, (cos_o, alpha, quad, mc)
            albedo[cos_o, alpha] = quad
        # plain GGX loses energy as the surface gets rougher (no multiple-scattering compensation) ...
        a = [albedo[cos_o, alpha] for alpha in ALPHAS]
        assert all(x >= y - 1e-3 for x, y in zip(a, a[1:])), a
        # ... and reflects all of it in the polished limit
        assert a[0] > 0.995, a


# ---- registers -------------------------------------------------------------------------------------------------------------
def test_metal_kernel_registers(rtb):
    """the metal kernels (k_shade's MODE 6 / 7 as k_shade_metal) are quoted in DESIGN.md and spill no more than the k_shade
    instantiation each extends (MODE 3 / 5, the same INLINE form)"""
    import importlib.util
    import re

    spec = importlib.util.spec_from_file_location("shade_regs", os.path.join(ROOT, "tools", "shade_regs.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    base = {name: row for name, *row in mod.table()}
    metal = {name: row for name, *row in mod.table(kernels=mod.METAL_KERNELS)}
    assert sorted(metal) == [f"k_shade_metal<{m}, {t}>" for m in (6, 7) for t in ("false", "true")], sorted(metal)
    design = open(os.path.join(ROOT, "DESIGN.md")).read()
    for name, (reg, stack, st, ld) in metal.items():
        assert re.search(re.escape(name) + r"\s+%d\s+%d\s+%d\s+%d" % (reg, stack, st, ld), design), name
        m, inline = name[len("k_shade_metal<")], name.endswith("true>")
        ref = base[f"k_shade<{3 if m == '6' else 5}, 0, 0, true, 256, {'true' if inline else 'false'}>"]
        assert st <= ref[2] and ld <= ref[3], (name, ref)
