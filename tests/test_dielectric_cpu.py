"""The dielectric material (brdf 3) without a GPU: the loader on host-only handles, the mesh orientation rule, the
Snell / Fresnel header (csrc/dielectric_rule.cuh) against a numpy restatement, and the f64 oracle against a closed form."""
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT

NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")


@pytest.fixture(scope="module")
def glass(oracle_mod):
    """the f64 oracle with the dielectric (tests/glass_oracle.py); oracle_mod builds the oracle whose entry points it shares"""
    import glass_oracle

    glass_oracle.lib()
    return glass_oracle

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


def scene(brdf, geometry="{ type = \"sphere\", pos = [0.0, 0.0, 0.0], r = 1.0 }", transforms=""):
    return CAMERA + LIGHT + f"""
[[objects]]
brdf = {brdf}
geometry = {geometry}
{transforms}
"""


def load(rtb, text, assets=None):
    return rtb.Scene.from_toml_string(text, assets_dir=assets, device=-1)


# ---- loader --------------------------------------------------------------------------------------------------------------
def test_toml_fields(rtb):
    o = load(rtb, scene('{ type = "dielectric", ior = 1.5, tint = [0.9, 0.5, 0.25] }')).object(1)
    assert o["brdf"] == 3 and o["k"] == [1.5, 1.0, 0.0] and o["color_d"] == [0.9, 0.5, 0.25]
    o = load(rtb, scene('{ type = "dielectric", ior = 1.33 }')).object(1)
    assert o["k"][0] == 1.33 and o["color_d"] == [1.0, 1.0, 1.0]       # tint defaults to 1


@pytest.mark.parametrize("brdf, field", [
    ('{ type = "dielectric" }', "ior"),
    ('{ type = "dielectric", ior = 0.0 }', "ior"),
    ('{ type = "dielectric", ior = -1.5 }', "ior"),
    ('{ type = "dielectric", ior = inf }', "ior"),
    ('{ type = "dielectric", ior = nan }', "ior"),
    ('{ type = "dielectric", ior = "glass" }', "ior"),
    ('{ type = "dielectric", ior = 1.5, tint = [1.0, 1.5, 1.0] }', "tint"),
    ('{ type = "dielectric", ior = 1.5, tint = [-0.1, 1.0, 1.0] }', "tint"),
    ('{ type = "dielectric", ior = 1.5, tint = [1.0, 1.0] }', "tint"),
])
def test_invalid_fields_name_the_field(rtb, brdf, field):
    with pytest.raises(rtb.LoadTomlError) as e:
        load(rtb, scene(brdf))
    assert e.value.code == rtb.RTB_EPARSE and field in str(e.value)


def test_unknown_variant_lists_dielectric(rtb):
    with pytest.raises(rtb.LoadTomlError) as e:
        load(rtb, scene('{ type = "glass", ior = 1.5 }'))
    assert e.value.code == rtb.RTB_EPARSE and "`dielectric`" in str(e.value)


def _objects(brdf):
    return [
        {"emitted": (4.0, 4.0, 4.0), "brdf": ("diffuse", (0.0, 0.0, 0.0)), "geometry": ("sphere", (0.0, 5.0, 0.0), 1.0)},
        {"brdf": brdf, "geometry": ("sphere", (0.0, 0.0, 0.0), 1.0)},
    ]


def test_scene_create_and_object_round_trip(rtb):
    sc = rtb.Scene.from_objects((0, 0, 10), (0, 0, -1), _objects(("dielectric", 1.5, (0.8, 0.6, 0.4))), device=-1)
    o = sc.object(1)
    assert o["brdf"] == 3 and o["k"] == [1.5, 1.0, 0.0] and o["color_d"] == pytest.approx([0.8, 0.6, 0.4])
    # what rtb_scene_object reports builds the same object again
    again = rtb.Scene.from_objects((0, 0, 10), (0, 0, -1), _objects(("dielectric", o["k"][0], o["color_d"])), device=-1).object(1)
    assert again == o
    assert rtb.Scene.from_objects((0, 0, 10), (0, 0, -1), _objects(("dielectric", 1.5)), device=-1).object(1)["color_d"] == [1.0, 1.0, 1.0]
    for bad in (("dielectric", 0.0), ("dielectric", float("nan")), ("dielectric", 1.5, (1.0, 2.0, 1.0))):
        with pytest.raises(rtb.LoadTomlError) as e:
            rtb.Scene.from_objects((0, 0, 10), (0, 0, -1), _objects(bad), device=-1)
        assert e.value.code == rtb.RTB_EPARSE and "dielectric" in str(e.value)


# ---- which side is outside -------------------------------------------------------------------------------------------------
TETRA_V = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [0, 0, 1]], float)
TETRA_F = [(1, 3, 2), (1, 2, 4), (1, 4, 3), (2, 3, 4)]      # counter-clockwise seen from outside: (b-a) x (c-a) points out


def _obj_file(path, faces):
    with open(path, "w") as f:
        for v in TETRA_V:
            f.write("v %g %g %g\n" % tuple(v))
        for fa in faces:
            f.write("f %d %d %d\n" % fa)


def _stored_normals_point_out(tris):
    c = tris.reshape(-1, 3).mean(0)
    a, b, cc = tris[:, 0].astype(np.float64), tris[:, 1].astype(np.float64), tris[:, 2].astype(np.float64)
    n = np.cross(cc - a, b - a)
    return np.sign(np.einsum("ij,ij->i", n, (a + b + cc) / 3 - c))


@pytest.mark.parametrize("geometry", ['{ type = "cube", pos = [-1.0, -1.0, -1.0], size = 2.0 }',
                                      '{ type = "prism", pos = [-1.0, -0.5, -2.0], size = [2.0, 1.0, 4.0] }'])
def test_builtin_meshes_are_oriented(rtb, glass, geometry):
    # the reference's prism winds one triangle of each face one way and the other the opposite way: the loader turns the
    # second kind around, so that every stored normal of the glass points the same way — out, as the first one does
    text = scene('{ type = "dielectric", ior = 1.5 }', geometry, "transforms = [ { rotate_y = 0.3 } ]")
    sc = load(rtb, text)
    assert sc.object(1)["k"][1] == 1.0
    tris = sc.triangles()
    assert (_stored_normals_point_out(tris) == 1).all()
    plain = load(rtb, text.replace('{ type = "dielectric", ior = 1.5 }', '{ type = "diffuse", kd = [0.5, 0.5, 0.5] }')).triangles()
    assert sorted(_stored_normals_point_out(plain)) == [-1] * 6 + [1] * 6     # the layout a diffuse prism keeps
    assert np.array_equal(tris, glass.OracleScene.from_toml_string(text).mesh_triangles(1).astype(np.float32))


@pytest.mark.parametrize("faces, sign", [(TETRA_F, -1.0), ([(a, c, b) for a, b, c in TETRA_F], 1.0)])
def test_obj_orientation_follows_the_winding(rtb, glass, tmp_path, faces, sign):
    # counter-clockwise faces seen from outside: the stored normal (c-a) x (b-a) points in, sign -1; the reversed file: +1
    _obj_file(tmp_path / "t.obj", faces)
    text = scene('{ type = "dielectric", ior = 1.5 }', '{ type = "mesh", path = "t.obj" }',
                 "transforms = [ { translate = [0.5, 0.0, 0.0] }, { scale = 3.0 } ]")
    sc = load(rtb, text, str(tmp_path))
    assert sc.object(1)["k"][1] == sign
    tris = sc.triangles()
    assert (_stored_normals_point_out(tris) == sign).all()
    assert np.array_equal(tris, glass.OracleScene.from_toml_string(text, str(tmp_path)).mesh_triangles(1).astype(np.float32))
    # one triangle of the file turned around: it is turned back, the sign is that of the first triangle
    mixed = [faces[0], faces[1], (faces[2][0], faces[2][2], faces[2][1]), faces[3]]
    _obj_file(tmp_path / "t.obj", mixed)
    sc = load(rtb, text, str(tmp_path))
    assert sc.object(1)["k"][1] == sign and (_stored_normals_point_out(sc.triangles()) == sign).all()


def test_scene_create_mesh_soup_is_oriented(rtb):
    # rtb_scene_create gives every triangle its own three vertices: pieces are joined by vertex POSITION
    tris = np.array([[TETRA_V[a - 1], TETRA_V[b - 1], TETRA_V[c - 1]] for a, b, c in TETRA_F[:2] + [(1, 3, 4), TETRA_F[3]]], np.float32)
    obs = _objects(("dielectric", 1.5))
    obs[1]["geometry"] = ("mesh", tris)
    sc = rtb.Scene.from_objects((0, 0, 10), (0, 0, -1), obs, device=-1)
    assert sc.object(1)["k"][1] == -1.0 and (_stored_normals_point_out(sc.triangles()) == -1).all()


# ---- the rule itself (csrc/dielectric_rule.cuh) ----------------------------------------------------------------------------
HARNESS = r"""
#include <cstdio>
#include "dielectric_rule.cuh"
using namespace rtb;
// stdin: n, then n records {dir xyz, nf xyz, flipped, orient, ior, u}; stdout: n records {dir xyz, refracted, F, cos_t, entering}
int main() {
    int n;
    if (fread(&n, 4, 1, stdin) != 1) return 1;
    for (int i = 0; i < n; ++i) {
        float r[10];
        if (fread(r, 4, 10, stdin) != 10) return 1;
        const float3 d = make_float3(r[0], r[1], r[2]), nf = make_float3(r[3], r[4], r[5]);
        const bool flipped = r[6] != 0.0f, entering = dielectric_entering(flipped, r[7]);
        bool refracted;
        const float3 o = dielectric_scatter(d, nf, flipped, r[7], r[8], r[9], refracted);
        float cos_t;
        const float F = dielectric_fresnel(-dot(d, nf), entering ? 1.0f / r[8] : r[8], cos_t);
        const float out[7] = {o.x, o.y, o.z, refracted ? 1.0f : 0.0f, F, cos_t, entering ? 1.0f : 0.0f};
        fwrite(out, 4, 7, stdout);
    }
    return 0;
}
"""


@pytest.fixture(scope="module")
def rule(tmp_path_factory):
    d = tmp_path_factory.mktemp("dielectric_rule")
    (d / "h.cu").write_text(HARNESS)
    exe = d / "h"
    subprocess.run([NVCC, "-std=c++17", "-O2", "-ccbin", "/usr/bin/g++", "-I", os.path.join(ROOT, "raytracer-server_b200", "csrc"),
                    str(d / "h.cu"), "-o", str(exe)], check=True)

    def run(d, nf, flipped, orient, ior, u):
        n = len(d)
        rec = np.concatenate([d, nf, np.stack([flipped, orient, ior, u], 1)], 1).astype(np.float32)
        out = subprocess.run([str(exe)], input=np.int32(n).tobytes() + rec.tobytes(), capture_output=True, check=True).stdout
        o = np.frombuffer(out, np.float32).reshape(n, 7).astype(np.float64)
        return {"dir": o[:, :3], "refracted": o[:, 3] == 1, "F": o[:, 4], "cos_t": o[:, 5], "entering": o[:, 6] == 1}

    return run


def fresnel_np(cos_i, eta):
    """the exact unpolarised Fresnel reflectance, (r_s^2 + r_p^2) / 2; 1 beyond the critical angle (in the inputs' precision)"""
    one = cos_i.dtype.type(1)
    sin2t = eta * eta * (one - cos_i * cos_i)
    tir = sin2t >= one
    cos_t = np.sqrt(np.clip(one - sin2t, 0, None))
    rs = (eta * cos_i - cos_t) / (eta * cos_i + cos_t)
    rp = (cos_i - eta * cos_t) / (cos_i + eta * cos_t)
    return np.where(tir, one, cos_i.dtype.type(0.5) * (rs * rs + rp * rp)), np.where(tir, cos_i.dtype.type(0), cos_t)


def _rays(rng, n):
    nf = rng.normal(size=(n, 3))
    nf /= np.linalg.norm(nf, axis=1, keepdims=True)
    d = rng.normal(size=(n, 3))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    d = np.where((np.einsum("ij,ij->i", d, nf) > 0)[:, None], -d, d)      # arriving against the facing normal
    return d.astype(np.float32).astype(np.float64), nf.astype(np.float32).astype(np.float64)


def test_rule_against_numpy(rule):
    rng = np.random.default_rng(5)
    n = 4000
    d, nf = _rays(rng, n)
    flipped, orient = rng.integers(0, 2, n), rng.choice([-1.0, 1.0], n)
    ior, u = rng.uniform(1.05, 2.4, n), rng.random(n)
    r = rule(d, nf, flipped, orient, ior, u)
    entering = (flipped == 0) != (orient < 0)
    assert (r["entering"] == entering).all()
    # the restatement in the header's fp32 arithmetic, operation for operation
    f32 = np.float32
    d32, n32, ior32 = d.astype(f32), nf.astype(f32), ior.astype(f32)
    eta = np.where(entering, f32(1) / ior32, ior32)
    cos_i = -(d32[:, 0] * n32[:, 0] + d32[:, 1] * n32[:, 1] + d32[:, 2] * n32[:, 2])
    F, cos_t = fresnel_np(cos_i, eta)
    assert np.abs(r["F"] - F).max() < 1e-6 and np.abs(r["cos_t"] - cos_t).max() < 1e-6
    eta, cos_i, F, cos_t = (x.astype(np.float64) for x in (eta, cos_i, F, cos_t))
    near = np.abs(u - F) < 1e-5                                              # fp32 vs f64 decides differently only at u == F
    assert (r["refracted"][~near] == (u >= F)[~near]).all()
    refl = d + 2 * cos_i[:, None] * nf
    refr = eta[:, None] * d + (eta * cos_i - cos_t)[:, None] * nf
    want = np.where(r["refracted"][:, None], refr, refl)
    assert np.abs(r["dir"] - want).max() < 1e-6
    assert np.abs(np.linalg.norm(r["dir"], axis=1) - 1).max() < 1e-6      # unit length
    t = r["refracted"]
    # Snell: |eta sin_i| = sin_t, and the transmitted ray goes through the surface
    sin_i = np.sqrt(np.clip(1 - cos_i ** 2, 0, None))
    sin_t = np.linalg.norm(np.cross(r["dir"], nf), axis=1)
    assert np.abs(eta[t] * sin_i[t] - sin_t[t]).max() < 1e-5       # an identity of the fp32 outputs, so a little looser
    assert (np.einsum("ij,ij->i", r["dir"][t], nf[t]) < 0).all() and (np.einsum("ij,ij->i", r["dir"][~t], nf[~t]) > 0).all()


def test_fresnel_limits_and_symmetry(rule):
    rng = np.random.default_rng(6)
    ior = np.array([1.33, 1.5, 2.0, 2.4])
    # normal incidence: ((ior - 1) / (ior + 1))^2, from either side
    nf = np.tile([[0.0, 0.0, 1.0]], (4, 1))
    d = -nf
    for flipped in (0, 1):
        r = rule(d, nf, np.full(4, flipped), np.ones(4), ior, np.full(4, 0.5))
        assert np.abs(r["F"] - ((ior - 1) / (ior + 1)) ** 2).max() < 1e-6
    # beyond the critical angle from inside: F = 1 and the ray is always reflected
    n = 500
    ior_r = rng.uniform(1.2, 2.4, n)
    theta = np.arcsin(1 / ior_r) + rng.uniform(1e-3, 1.0, n) * (np.pi / 2 - np.arcsin(1 / ior_r))
    d = np.stack([np.sin(theta), np.zeros(n), -np.cos(theta)], 1)
    r = rule(d, np.tile([[0.0, 0.0, 1.0]], (n, 1)), np.ones(n), np.ones(n), ior_r, np.full(n, 0.999999))
    assert (r["F"] == 1).all() and not r["refracted"].any()
    # the same interface seen from the other side at the corresponding (refracted) angle reflects the same fraction
    theta_i = rng.uniform(0, 1.5, n)
    ior_s = rng.uniform(1.1, 2.4, n)
    theta_t = np.arcsin(np.sin(theta_i) / ior_s)
    z = np.tile([[0.0, 0.0, 1.0]], (n, 1))
    out = rule(np.stack([np.sin(theta_i), np.zeros(n), -np.cos(theta_i)], 1), z, np.zeros(n), np.ones(n), ior_s, np.full(n, 0.5))
    back = rule(np.stack([np.sin(theta_t), np.zeros(n), -np.cos(theta_t)], 1), z, np.ones(n), np.ones(n), ior_s, np.full(n, 0.5))
    assert np.abs(out["F"] - back["F"]).max() < 1e-5


def test_entering_truth_table(rule):
    f = np.array([0, 1, 0, 1])
    s = np.array([1.0, 1.0, -1.0, -1.0])
    r = rule(np.tile([[0.0, 0.0, -1.0]], (4, 1)), np.tile([[0.0, 0.0, 1.0]], (4, 1)), f, s, np.full(4, 1.5), np.full(4, 0.5))
    assert list(r["entering"]) == [True, False, False, True]


# ---- the oracle against a closed form --------------------------------------------------------------------------------------
# A camera ray through the centre of a glass sphere towards a large emitter behind it: the internal reflections run along the
# axis, what leaves towards the camera sees black, so L = Le * T^2 * (1 + R^2 + R^4 + ...) = Le * (1 - F0) / (1 + F0).
AXIS_SCENE = """
[camera]
pos = [0.0, 0.0, 10.0]
dir = [0.0, 0.0, -1.0]
[[objects]]
emitted = [1.0, 0.5, 0.25]
brdf = { type = "diffuse", kd = [0.0, 0.0, 0.0] }
geometry = { type = "sphere", pos = [0.0, 0.0, -1000.0], r = 900.0 }
[[objects]]
brdf = { type = "dielectric", ior = 1.5 }
geometry = { type = "sphere", pos = [0.0, 0.0, 0.0], r = 1.0 }
"""
AXIS_W = 2001                                  # pixel 1000 of a 2001 x 2001 frame looks down the axis to within 0.6 mrad
AXIS_WANT = np.array([1.0, 0.5, 0.25]) * (1 - 0.04) / (1 + 0.04)


def test_oracle_transmittance_closed_form(glass):
    o = glass.OracleScene.from_toml_string(AXIS_SCENE)
    n = 60000
    L = o.sample_radiance(AXIS_W, AXIS_W, 4 * n, 3, np.full(n, 1000), np.full(n, 1000), np.arange(n) * 4)
    assert np.abs(L.mean(0) / AXIS_WANT - 1).max() < 0.01, L.mean(0)
