"""Next-event estimation over every emitter (EST_NEE_ALL_LIGHTS) without a GPU: the light table on host-only handles against a
numpy f64 restatement, the selection / triangle-point / weight header (csrc/light_rule.cuh) against numpy, the f64 oracle's
estimator 3 against estimator 0 and against closed-form form factors, the server's "all_lights" field, and the register table
of the new k_shade instantiations."""
import importlib.util
import os
import re
import subprocess

import numpy as np
import pytest

from conftest import ROOT, SCENES, scene_path

NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
LUM = np.array([0.2126, 0.7152, 0.0722])


@pytest.fixture(scope="module")
def oracle3(oracle_mod):
    """the f64 glass oracle with estimator 3 (tests/lights_oracle.py); oracle_mod builds the oracle whose entry points it shares"""
    import lights_oracle

    lights_oracle.lib()
    return lights_oracle


CAMERA = """
[camera]
pos = [0.0, 0.0, 10.0]
dir = [0.0, 0.0, -1.0]
"""


def obj(emitted, geometry, transforms="", brdf='{ type = "diffuse", kd = [0.0, 0.0, 0.0] }'):
    return f"""
[[objects]]
emitted = {list(map(float, emitted))}
brdf = {brdf}
geometry = {geometry}
{transforms}
"""


def load(rtb, text, assets=None):
    return rtb.Scene.from_toml_string(text, assets_dir=assets, device=-1)


def _rot(axis, a):
    c, s = np.cos(a), np.sin(a)
    return {0: np.array([[1, 0, 0], [0, c, -s], [0, s, c]]), 1: np.array([[c, 0, s], [0, 1, 0], [-s, 0, c]]),
            2: np.array([[c, -s, 0], [s, c, 0], [0, 0, 1]])}[axis]


def _true_area(tris):
    t = np.asarray(tris, np.float64)
    return 0.5 * np.linalg.norm(np.cross(t[:, 1] - t[:, 0], t[:, 2] - t[:, 0]), axis=1).sum()


def _want(emitted_area):
    """(objects, prob) of the table for [(object, emitted, area)] in object order"""
    w = np.array([max(0.0, float(LUM @ np.maximum(e, 0))) * a for _, e, a in emitted_area])
    keep = w > 0
    return np.array([o for o, _, _ in emitted_area])[keep], w[keep] / w[keep].sum()


# ---- the light table --------------------------------------------------------------------------------------------------------
def test_spheres(rtb):
    spheres = [((50.0, 50.0, 50.0), (0.0, 5.0, 0.0), 1.0, ""), ((0.0, 8.0, 2.0), (3.0, 0.0, 0.0), 0.5, "transforms = [ { scale = 3.0 } ]"),
               ((1.0, 0.0, 0.0), (-3.0, 0.0, 0.0), 2.0, ""), ((0.0, 0.0, 0.0), (0.0, -3.0, 0.0), 1.0, "")]
    text = CAMERA + "".join(obj(e, f'{{ type = "sphere", pos = {list(p)}, r = {r} }}', t) for e, p, r, t in spheres)
    L = load(rtb, text).lights()
    radii = [1.0, 1.5, 2.0, 1.0]
    objs, prob = _want([(i, np.array(e), 4 * np.pi * r * r) for i, ((e, _, _, _), r) in enumerate(zip(spheres, radii))])
    assert list(L["objects"]) == list(objs) == [0, 1, 2]
    np.testing.assert_allclose(L["prob"], prob, rtol=1e-12)
    np.testing.assert_allclose(L["area"], [4 * np.pi * r * r for r in radii[:3]], rtol=1e-12)
    assert abs(L["prob"].sum() - 1) < 1e-12


def test_mesh_lights_use_the_true_area(rtb, tmp_path):
    # the built-in cube, scaled and rotated: Mesh::surface_area is that of the untransformed cube (24), the table's is 24 * 2.5^2
    (tmp_path / "quad.obj").write_text("v 0 0 0\nv 2 0 0\nv 2 0 1\nv 0 0 1\nf 1 2 3\nf 1 3 4\n")
    text = (CAMERA + obj((4.0, 4.0, 4.0), '{ type = "sphere", pos = [0.0, 5.0, 0.0], r = 0.5 }') +
            obj((1.0, 2.0, 0.5), '{ type = "cube", pos = [-1.0, -1.0, -1.0], size = 2.0 }',
                "transforms = [ { scale = 2.5 }, { rotate_y = 0.7 }, { rotate_x = -0.3 }, { translate = [1.0, 0.0, 0.0] } ]") +
            obj((0.0, 0.0, 3.0), '{ type = "mesh", path = "quad.obj" }', "transforms = [ { rotate_z = 1.1 }, { scale = 0.5 } ]"))
    sc = load(rtb, text, str(tmp_path))
    assert sc.object(1)["surface_area"] == pytest.approx(24.0)
    tris = sc.triangles().astype(np.float64)
    cube, quad = tris[sc.object(1)["first_triangle"]:][:12], tris[sc.object(2)["first_triangle"]:][:2]
    assert _true_area(cube) == pytest.approx(24 * 2.5 ** 2, rel=1e-6)
    assert _true_area(quad) == pytest.approx(2 * 0.5 ** 2, rel=1e-6)
    L = sc.lights()
    objs, prob = _want([(0, np.array([4.0, 4, 4]), np.pi), (1, np.array([1.0, 2, 0.5]), 24 * 6.25), (2, np.array([0.0, 0, 3]), 0.5)])
    assert list(L["objects"]) == list(objs) == [0, 1, 2]
    np.testing.assert_allclose(L["area"], [np.pi, 24 * 6.25, 0.5], rtol=1e-12)
    np.testing.assert_allclose(L["prob"], prob, rtol=1e-12)
    # the f64 restatement from the object's own vertices (the loader's transforms, not a re-derivation here)
    cube0 = np.array([[0, 0, 0], [0, 0, 2], [0, 2, 0], [0, 2, 2], [2, 0, 0], [2, 0, 2], [2, 2, 0], [2, 2, 2]], float) - 1.0
    c = cube0.mean(0)
    v = c + (cube0 - c) * 2.5
    v = (v - v.mean(0)) @ _rot(1, 0.7).T + v.mean(0)
    assert _true_area(v[np.array([1, 3, 7, 1, 5, 7, 0, 2, 6, 0, 4, 6, 0, 1, 3, 0, 2, 3, 4, 5, 7, 4, 6, 7, 2, 3, 7, 2, 6, 7, 0, 1, 5, 0, 4, 5]).reshape(12, 3)]) \
        == pytest.approx(L["area"][1], rel=1e-12)


def test_planes_and_zero_weight_emitters_stay_out(rtb):
    text = (CAMERA + obj((10.0, 10.0, 10.0), '{ type = "sphere", pos = [0.0, 5.0, 0.0], r = 1.0 }') +
            obj((5.0, 5.0, 5.0), '{ type = "plane", pos = [0.0, -1.0, 0.0], n = [0.0, 1.0, 0.0] }') +
            obj((-3.0, 0.0, 0.0), '{ type = "sphere", pos = [2.0, 0.0, 0.0], r = 1.0 }') +
            obj((1.0, 1.0, 1.0), '{ type = "sphere", pos = [-2.0, 0.0, 0.0], r = 0.0 }') +
            obj((0.0, 1.0, 0.0), '{ type = "sphere", pos = [-4.0, 0.0, 0.0], r = 0.25 }'))
    L = load(rtb, text).lights()
    assert list(L["objects"]) == [0, 4]
    np.testing.assert_allclose(L["prob"], _want([(0, np.array([10.0] * 3), 4 * np.pi), (4, np.array([0, 1.0, 0]), np.pi / 4)])[1], rtol=1e-12)
    assert abs(L["prob"].sum() - 1) < 1e-12


def test_table_survives_export_and_import(rtb):
    for name in ("cornell_box", "cubes", "flying_unicorn"):
        sc = rtb.Scene.from_toml(scene_path(name), device=-1)
        L, again = sc.lights(), rtb.Scene.from_export(sc.export(), device=-1).lights()
        assert list(L["objects"]) == [sc.light_source] and L["prob"][0] == 1.0
        for k in L:
            assert np.array_equal(L[k], again[k])


# ---- the rule itself (csrc/light_rule.cuh) -----------------------------------------------------------------------------------
HARNESS = r"""
#include <cstdio>
#include <vector>
#include "light_rule.cuh"
using namespace rtb;
// stdin: n_cdf, cdf[n_cdf], n, then n records {u, a xyz, b xyz, c xyz, u1, u2, nf xyz, w xyz, r2, pdf_area}
// stdout: n records {pick, point xyz, normal xyz, weight}
int main() {
    int m, n;
    if (fread(&m, 4, 1, stdin) != 1) return 1;
    std::vector<float> cdf(m);
    if (fread(cdf.data(), 4, m, stdin) != (size_t)m || fread(&n, 4, 1, stdin) != 1) return 1;
    for (int i = 0; i < n; ++i) {
        float r[20];
        if (fread(r, 4, 20, stdin) != 20) return 1;
        auto v = [&](int k) { return make_float3(r[k], r[k + 1], r[k + 2]); };
        const float3 p = light_tri_point(v(1), v(4), v(7), r[10], r[11]);
        const float3 ny = light_tri_normal(v(1), v(4), v(7));
        const float out[8] = {(float)light_pick(cdf.data(), m, r[0]), p.x, p.y, p.z, ny.x, ny.y, ny.z, light_weight(v(12), ny, v(15), r[18], r[19])};
        fwrite(out, 4, 8, stdout);
    }
    return 0;
}
"""


@pytest.fixture(scope="module")
def rule(tmp_path_factory):
    d = tmp_path_factory.mktemp("light_rule")
    (d / "h.cu").write_text(HARNESS)
    exe = d / "h"
    subprocess.run([NVCC, "-std=c++17", "-O2", "-ccbin", "/usr/bin/g++", "-I", os.path.join(ROOT, "raytracer-server_b200", "csrc"),
                    str(d / "h.cu"), "-o", str(exe)], check=True)

    def run(cdf, rec):
        cdf = np.asarray(cdf, np.float32)
        rec = np.asarray(rec, np.float32)
        inp = np.int32(cdf.size).tobytes() + cdf.tobytes() + np.int32(len(rec)).tobytes() + rec.tobytes()
        o = np.frombuffer(subprocess.run([str(exe)], input=inp, capture_output=True, check=True).stdout, np.float32).reshape(-1, 8)
        return o[:, 0].astype(int), o[:, 1:4].astype(np.float64), o[:, 4:7].astype(np.float64), o[:, 7].astype(np.float64)

    return run


def test_rule_against_numpy(rule):
    rng = np.random.default_rng(11)
    n = 5000
    w = rng.random(7)
    w[3] = 0.0                                                    # a zero-weight entry is never picked
    cdf = np.cumsum(w) / w.sum()
    cdf[-1] = 1.0
    tri = rng.normal(size=(n, 3, 3))
    u1, u2, u = rng.random(n), rng.random(n), rng.random(n)
    nf = rng.normal(size=(n, 3))
    nf /= np.linalg.norm(nf, axis=1, keepdims=True)
    wd = rng.normal(size=(n, 3))
    wd /= np.linalg.norm(wd, axis=1, keepdims=True)
    r2, pdf = rng.uniform(0.5, 20, n), rng.uniform(0.01, 2, n)
    rec = np.concatenate([u[:, None], tri.reshape(n, 9), u1[:, None], u2[:, None], nf, wd, r2[:, None], pdf[:, None]], 1)
    rec32 = rec.astype(np.float32).astype(np.float64)
    pick, p, ny, weight = rule(cdf, rec)
    # selection: partition_point(cdf <= u), clamped (the fp32 values the header sees)
    cdf32 = cdf.astype(np.float32)
    want = np.minimum(np.searchsorted(cdf32, rec32[:, 0].astype(np.float32), side="right"), len(cdf) - 1)
    assert (pick == want).all() and not (pick == 3).any()
    assert (rule(cdf, np.concatenate([[[1.0]], rec[:1, 1:]], 1))[0] == 6).all()          # u beyond the last entry: the last one
    # the point: (1 - sqrt u1) a + sqrt u1 (1 - u2) b + sqrt u1 u2 c, inside the triangle
    a, b, c = rec32[:, 1:4], rec32[:, 4:7], rec32[:, 7:10]
    s = np.sqrt(rec32[:, 10])[:, None]
    bary = np.stack([1 - s[:, 0], s[:, 0] * (1 - rec32[:, 11]), s[:, 0] * rec32[:, 11]], 1)
    assert (bary >= 0).all() and np.allclose(bary.sum(1), 1)
    np.testing.assert_allclose(p, (1 - s) * a + s * (1 - rec32[:, 11:12]) * b + s * rec32[:, 11:12] * c, atol=1e-6 * (1 + np.abs(tri).max()))
    nrm = np.cross(c - a, b - a)
    np.testing.assert_allclose(ny, nrm / np.linalg.norm(nrm, axis=1, keepdims=True), atol=3e-6)   # fp32 cross product + rsqrt
    # the weight: max(n_f . w, 0) |n_y . w| / (r2 pdf)
    nfv, wv = rec32[:, 12:15], rec32[:, 15:18]
    want_w = np.maximum(np.einsum("ij,ij->i", nfv, wv), 0) * np.abs(np.einsum("ij,ij->i", ny, wv)) / (rec32[:, 18] * rec32[:, 19])
    np.testing.assert_allclose(weight, want_w, rtol=1e-6, atol=1e-6)
    assert (weight[np.einsum("ij,ij->i", nfv, wv) < 0] == 0).all()


def test_uniform_points_cover_the_triangle(rule):
    # barycentric coordinates of the sampled points: uniform over the triangle (the mean is the centroid, the share of the
    # sub-triangle towards each vertex is 1/4)
    rng = np.random.default_rng(12)
    n = 40000
    tri = np.array([[0.0, 0, 0], [3, 0, 0], [0, 2, 0]])
    rec = np.zeros((n, 20))
    rec[:, 0] = 0.5
    rec[:, 1:10] = tri.reshape(9)
    rec[:, 10], rec[:, 11] = rng.random(n), rng.random(n)
    rec[:, 12:15] = rec[:, 15:18] = [0, 0, 1]
    rec[:, 18:20] = 1
    _, p, _, _ = rule([1.0], rec)
    np.testing.assert_allclose(p.mean(0), tri.mean(0), atol=0.02)
    corner = (p[:, 0] / 3 + p[:, 1] / 2) < 0.5                        # the half-size triangle at vertex a
    assert abs(corner.mean() - 0.25) < 0.01


# ---- the oracle ----------------------------------------------------------------------------------------------------------------
def test_oracle_single_sphere_light_equals_nee(oracle3):
    # rule 6 of DESIGN §3f: with one sphere light the estimators agree path by path, but where the reference's unclamped cosine
    # is negative and the shadow test still passes (about one path in 1500 here, by < 2e-6).  Estimator 3 drops that negative
    # term, so it is never below estimator 0.
    W, H = 600, 450
    rng = np.random.default_rng(21)
    n = 3000
    px, py, si = rng.integers(0, W, n), rng.integers(0, H, n), rng.integers(0, 64, n)
    for name in ("cornell_box", "cubes", "flying_unicorn"):
        o = oracle3.OracleScene.from_toml_string(open(scene_path(name)).read(), os.path.join(SCENES, "assets"))
        o.set_modes(oracle3.ACCEL_EXACT, 0)
        nee = o.sample_radiance(W, H, 64, 7, px, py, si)
        o.set_modes(oracle3.ACCEL_EXACT, 3)
        alll = o.sample_radiance(W, H, 64, 7, px, py, si)
        d = alll - nee
        assert (np.abs(d).max(1) <= 1e-12 * (1 + np.abs(nee).max())).mean() >= 0.998, name
        assert d.min() > -1e-12 and d.max() < 1e-5, name
        assert np.abs(nee).sum() > 0


# a floor (kd 0.5) lit by a 1 x 1 two-triangle rectangle 2 above the floor point and a sphere off to the side; nothing else
# reflects, so the radiance at the floor point is kd (Le1 F1 + Le2 F2) with the closed-form form factors
FF_H, FF_A, FF_C, FF_R, FF_KD = 2.0, 0.5, np.array([3.0, 2.0, 0.0]), 0.5, 0.5
FF_LE1, FF_LE2 = np.array([3.0, 2.0, 1.0]), np.array([1.0, 4.0, 8.0])


def _ff_scene(tmp_path):
    (tmp_path / "rect.obj").write_text(f"v {-FF_A} {FF_H} {-FF_A}\nv {FF_A} {FF_H} {-FF_A}\nv {FF_A} {FF_H} {FF_A}\nv {-FF_A} {FF_H} {FF_A}\n"
                                       "f 1 2 3\nf 1 3 4\n")
    return f"""
[camera]
pos = [0.0, 1.0, 0.0]
dir = [0.0, -1.0, 0.0]
[[objects]]
emitted = {[float(x) for x in FF_LE1]}
brdf = {{ type = "diffuse", kd = [0.0, 0.0, 0.0] }}
geometry = {{ type = "mesh", path = "rect.obj" }}
[[objects]]
emitted = {[float(x) for x in FF_LE2]}
brdf = {{ type = "diffuse", kd = [0.0, 0.0, 0.0] }}
geometry = {{ type = "sphere", pos = {[float(x) for x in FF_C]}, r = {FF_R} }}
[[objects]]
brdf = {{ type = "diffuse", kd = [{FF_KD}, {FF_KD}, {FF_KD}] }}
geometry = {{ type = "plane", pos = [0.0, 0.0, 0.0], n = [0.0, 1.0, 0.0] }}
"""


def _ff_rect_corner(a, b, h):
    """point to a parallel a x b rectangle at height h whose corner lies straight above the point"""
    A, B = a / h, b / h
    return (A / np.sqrt(1 + A * A) * np.arctan(B / np.sqrt(1 + A * A)) + B / np.sqrt(1 + B * B) * np.arctan(A / np.sqrt(1 + B * B))) / (2 * np.pi)


def test_oracle_two_lights_closed_form(oracle3, tmp_path):
    o = oracle3.OracleScene.from_toml_string(_ff_scene(tmp_path), str(tmp_path))
    o.set_modes(oracle3.ACCEL_EXACT, 3)
    F1 = 4 * _ff_rect_corner(FF_A, FF_A, FF_H)
    D = np.linalg.norm(FF_C)
    F2 = (FF_R / D) ** 2 * (FF_C[1] / D)                                 # a sphere wholly above the horizon
    want = FF_KD * (FF_LE1 * F1 + FF_LE2 * F2)
    n = 400000
    W = 2001                                                              # the centre pixel sees the floor point to within 0.3 mm
    L = o.sample_radiance(W, W, 4 * n, 5, np.full(n, 1000), np.full(n, 1000), np.arange(n) * 4)
    assert np.abs(L.mean(0) / want - 1).max() < 0.005, (L.mean(0), want)


# ---- server: "all_lights": true ----------------------------------------------------------------------------------------------
websockets = pytest.importorskip("websockets")


def test_all_lights_request_reaches_the_factory(rtb):
    from test_adaptive_cpu import _Job, _send, _serve

    calls = []

    def factory(scene, spp, passes=1, **kw):
        calls.append((scene, spp, passes, kw))
        return _Job()

    port, stop = _serve(factory)
    try:
        for req in [{"spp": 64, "all_lights": True}, {"spp": 64, "passes": 8, "all_lights": True, "denoise": True},
                    {"spp": 100, "noise": 2, "all_lights": True}, {"spp": 64, "all_lights": False}, {"spp": 64}]:
            assert _send(port, {"type": "render", "scene": "cornell_box", **req}) == bytes([0, 1, 0, 0, 0, 0, 1, 2, 3])
    finally:
        stop()
    assert calls == [("cornell_box", 64, 1, {"all_lights": True}), ("cornell_box", 64, 8, {"denoise": True, "all_lights": True}),
                     ("cornell_box", 96, 1, {"adaptive": {"target_levels": 2.0, "pass_spp": 16, "min_spp": 64}, "all_lights": True}),
                     ("cornell_box", 64, 1, {}), ("cornell_box", 64, 1, {})]


@pytest.mark.parametrize("value", ["true", 1, 0, None, [True], {"on": True}])
def test_bad_all_lights_closes_the_connection(rtb, value):
    from test_adaptive_cpu import _Job, _send, _serve

    calls = []
    port, stop = _serve(lambda *a, **kw: calls.append(a) or _Job())
    try:
        assert _send(port, {"type": "render", "scene": "cornell_box", "spp": 64, "all_lights": value}, expect_close=True) == 1007
    finally:
        stop()
    assert calls == []


# ---- the new k_shade instantiations (tools/shade_regs.py on the built engine.o) ------------------------------------------------
# the table the parent commit's build printed: the all-lights kernels leave every existing instantiation as it was
PARENT_ROWS = """
k_generate<0, 0>                       48      0         0         0
k_generate<5, 1>                       54      0         0         0
k_generate<5, 2>                       60      0         0         0
k_generate<5, 3>                       60      0         0         0
k_shade<0, 0, 0, true, 256, false>    128      8         4         8
k_shade<0, 0, 0, true, 256, true>     127    288        16        32
k_shade<1, 0, 0, true, 160, false>     93      0         0         0
k_shade<1, 0, 0, true, 160, true>      96    304        24        24
k_shade<1, 5, 1, true, 160, false>     93      0         0         0
k_shade<1, 5, 2, true, 160, false>     93      0         0         0
k_shade<1, 5, 3, false, 160, false>    95      0         0         0
k_shade<1, 5, 3, true, 160, false>     93      0         0         0
k_shade<1, 8, 0, true, 160, false>     93      0         0         0
k_shade<2, 0, 0, true, 256, false>    128      0         0         0
k_shade<2, 0, 0, true, 256, true>     125    288        12        24
k_shade<2, 5, 1, true, 256, false>    128      0         0         0
k_shade<2, 5, 2, true, 256, false>    128      0         0         0
k_shade<2, 5, 3, false, 160, false>    96     32        70        64
k_shade<2, 5, 3, true, 256, false>    128      0         0         0
k_shade<2, 8, 0, true, 256, false>    128      0         0         0
k_shade<3, 0, 0, true, 256, false>    128      8         4         8
k_shade<3, 0, 0, true, 256, true>     127    288        16        32
k_traverse<false>                      48    304        60        56
k_traverse<true>                       64    304        12        16
"""


def _rows():
    spec = importlib.util.spec_from_file_location("shade_regs", os.path.join(ROOT, "tools", "shade_regs.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return {name: (reg, stack, st, ld) for name, reg, stack, st, ld in mod.table()}


def test_register_table(rtb):
    rows = _rows()
    parent = {line[:36].strip(): tuple(int(x) for x in line[36:].split()) for line in PARENT_ROWS.strip().splitlines()}
    for name, nums in parent.items():
        assert rows.pop(name) == nums, name
    new = sorted(rows)
    assert new == ["k_shade<4, 0, 0, true, 256, false>", "k_shade<4, 0, 0, true, 256, true>",
                   "k_shade<5, 0, 0, true, 256, false>", "k_shade<5, 0, 0, true, 256, true>"]
    design = open(os.path.join(ROOT, "DESIGN.md")).read()
    for name in new:
        reg, stack, st, ld = rows[name]
        assert re.search(re.escape(name) + r"\s+%d\s+%d\s+%d\s+%d" % (reg, stack, st, ld), design), name
        # no more spill traffic than the kernel it extends (MODE 4: MODE 0, MODE 5: MODE 3)
        base = parent[("k_shade<0" if name.startswith("k_shade<4") else "k_shade<3") + name[len("k_shade<4"):]]
        assert st <= base[2] and ld <= base[3], name
