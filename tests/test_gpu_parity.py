"""Parity tests proper: the CUDA path (through the C ABI) against the oracle on the same inputs.

Gates from BASELINE.json: primary-ray first-hit ids bit-exact, hit distances within 1e-4 relative,
images within 1 % mean relative error per channel and PSNR >= 40 dB, estimator on ("MIS" dead branch)
and off (live NEE).  fp32-vs-f64 ambiguity: a ray whose f64 answer changes when its direction is
nudged by 2e-6 (about the fp32 rounding of a direction) sits on a silhouette / edge; such rays are
excluded from the bit-exact gate and their number is bounded.
"""
import os

import numpy as np
import pytest

from conftest import NCPU, SCENE_NAMES, SCENES, scene_path
from parity_metrics import channel_mre, path_error, pixel_mre, psnr

pytestmark = pytest.mark.gpu

T_REL_TOL = 1e-4          # BASELINE.json: "hit distances must match within 1e-4 relative"
ASSETS = os.path.join(SCENES, "assets")


def ambiguous_mask(osc, org, dirs, base, t_gpu=None):
    """rays whose oracle answer is unstable under a 2e-6 direction perturbation, or whose two candidate
    surfaces coincide (|t_gpu - t_oracle| <= 1e-5 t: e.g. the cubes' bottom faces lie IN the floor plane,
    scenes/cubes.toml; which of two coplanar primitives is 'nearer' is decided by rounding in f64 as well)"""
    amb = np.zeros(org.shape[0], dtype=bool)
    if t_gpu is not None:
        with np.errstate(invalid="ignore"):
            amb |= np.abs(t_gpu.astype(np.float64) - base["t"]) <= 1e-5 * np.abs(base["t"])
    rng = np.random.default_rng(0)
    for _ in range(4):
        d = dirs + rng.normal(scale=2e-6, size=dirs.shape)
        d /= np.linalg.norm(d, axis=1, keepdims=True)
        r = osc.trace_rays(org, d)
        amb |= (r["obj"] != base["obj"]) | (r["tri"] != base["tri"])
    return amb


@pytest.mark.parametrize("name", SCENE_NAMES)
@pytest.mark.parametrize("sub", [(0, 0, 0.0, 0.0), (1, 1, 0.3, -0.7)])
def test_primary_hits_bit_exact(gpu_scene, oracle_scene, parity_log, name, sub):
    W, H = 600, 450                       # the reference server's frame (src/server.rs:29-30)
    g, o = gpu_scene(name), oracle_scene(name)
    sx, sy, dx, dy = sub
    org, dirs = o.primary_rays(W, H, sx, sy, dx, dy)
    ro = o.trace_rays(org, dirs)
    rg = g.trace_primary(W, H, sx, sy, dx, dy)
    mism = (ro["obj"] != rg["obj"]) | (ro["tri"] != rg["tri"])
    n_unamb = 0
    if mism.any():
        idx = np.flatnonzero(mism)
        amb = ambiguous_mask(o, org[idx], dirs[idx], {k: v[idx] for k, v in ro.items()}, rg["t"][idx])
        n_unamb = int((~amb).sum())
    ok = ~mism & (ro["obj"] >= 0)
    rel = np.abs(rg["t"][ok].astype(np.float64) - ro["t"][ok]) / ro["t"][ok]
    parity_log(f"gpu/primary_ids/{name}/sub{sx}{sy}", rays=mism.size, mismatches=int(mism.sum()), unambiguous_mismatches=n_unamb,
               t_rel_max=rel.max(), t_rel_median=np.median(rel), mesh_hits=int((ro["tri"] >= 0).sum()))
    assert n_unamb == 0, f"{n_unamb} unambiguous primary rays got a different first hit"
    assert mism.mean() < 2e-4, f"too many ambiguous rays: {mism.sum()} of {mism.size}"
    assert rel.max() < T_REL_TOL
    assert (rg["obj"] != 5).all()         # duplicate wall: lowest object index wins (src/scene.rs:277-284)


@pytest.mark.parametrize("name", SCENE_NAMES)
def test_secondary_rays_match(gpu_scene, oracle_scene, parity_log, name):
    # incoherent rays from inside the room, the kind the integrator produces
    g, o = gpu_scene(name), oracle_scene(name)
    rng = np.random.default_rng(5)
    n = 200_000
    org = np.column_stack([rng.uniform(2, 98, n), rng.uniform(1, 80, n), rng.uniform(5, 250, n)])
    d = rng.normal(size=(n, 3))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    org32, d32 = org.astype(np.float32), d.astype(np.float32)
    d32 /= np.linalg.norm(d32.astype(np.float64), axis=1, keepdims=True).astype(np.float32)
    ro = o.trace_rays(org32.astype(np.float64), d32.astype(np.float64))   # identical (fp32-representable) rays
    rg = g.trace_rays(org32, d32)
    mism = (ro["obj"] != rg["obj"]) | (ro["tri"] != rg["tri"])
    n_unamb = 0
    if mism.any():
        idx = np.flatnonzero(mism)
        amb = ambiguous_mask(o, org32[idx].astype(np.float64), d32[idx].astype(np.float64), {k: v[idx] for k, v in ro.items()}, rg["t"][idx])
        n_unamb = int((~amb).sum())
    ok = ~mism & (ro["obj"] >= 0)
    rel = np.abs(rg["t"][ok].astype(np.float64) - ro["t"][ok]) / np.maximum(ro["t"][ok], 1e-3)
    parity_log(f"gpu/secondary_rays/{name}", rays=n, mismatches=int(mism.sum()), unambiguous_mismatches=n_unamb,
               t_rel_q9999=np.quantile(rel, 0.9999), t_rel_max=rel.max(), mesh_hits=int((ro["tri"] >= 0).sum()))
    assert n_unamb <= 2, f"{n_unamb} unambiguous rays differ"
    assert mism.mean() < 2e-3      # cubes: origins inside a cube see its bottom face and the floor at the same t
    assert np.quantile(rel, 0.9999) < T_REL_TOL


@pytest.mark.parametrize("name", SCENE_NAMES)
def test_fp32_oracle_explains_what_f64_cannot(gpu_scene, oracle_scene, oracle_f32_twin, parity_log, name):
    # SURVEY 8(f)4: an fp32 build of the oracle, fed with the GPU's own fp32 geometry, instead of excluding "ambiguous" rays.
    # For every ray, the GPU's answer must be the f64 oracle's or — where fp32 storage of the scene flips the reference's own
    # arithmetic — the fp32 oracle's; what neither explains may only be an exact distance tie between two surfaces.
    g, o, o32 = gpu_scene(name), oracle_scene(name), oracle_f32_twin(name)
    W, H = 600, 450
    org, dirs = o.primary_rays(W, H, 1, 0, 0.25, -0.4)
    rng = np.random.default_rng(21)
    n = 150_000
    so = np.column_stack([rng.uniform(2, 98, n), rng.uniform(1, 80, n), rng.uniform(5, 250, n)])
    sd = rng.normal(size=(n, 3))
    sd /= np.linalg.norm(sd, axis=1, keepdims=True)
    org32 = np.concatenate([org, so]).astype(np.float32)
    d32 = np.concatenate([dirs, sd]).astype(np.float32)
    d32 /= np.linalg.norm(d32.astype(np.float64), axis=1, keepdims=True).astype(np.float32)
    r64 = o.trace_rays(org32.astype(np.float64), d32.astype(np.float64))
    r32 = o32.trace_rays(org32, d32)
    rg = g.trace_rays(org32, d32)
    same = lambda a, b: (a["obj"] == b["obj"]) & (a["tri"] == b["tri"])   # noqa: E731
    by64, by32 = same(rg, r64), same(rg, r32)
    unexplained = ~by64 & ~by32
    with np.errstate(invalid="ignore"):
        tie = unexplained & (np.abs(rg["t"].astype(np.float64) - r64["t"]) <= 1e-5 * np.abs(r64["t"]))
    parity_log(f"gpu/fp32_oracle/{name}", rays=int(by64.size), f64_and_f32_oracles_differ=int((~same(r64, r32)).sum()), gpu_differs_from_f64=int((~by64).sum()),
               of_those_explained_by_f32_oracle=int((~by64 & by32).sum()), unexplained_exact_ties=int(tie.sum()), unexplained_other=int((unexplained & ~tie).sum()))
    assert (unexplained & ~tie).sum() <= 2
    assert (~by64).mean() < 2e-3


@pytest.mark.parametrize("mesh,n_tri", [("chair.obj", 212), ("crewmate.obj", 3412)])
def test_extra_meshes_lbvh(rtb, oracle_mod, mesh, n_tri):
    # the reference's unused assets as additional LBVH cases (SURVEY §8f rank 2)
    text = f"""
[camera]
pos = [0.0, 1.0, 6.0]
dir = [0.0, -0.1, -1.0]
[[objects]]
brdf = {{ type = "diffuse", kd = [0.7, 0.7, 0.7] }}
geometry = {{ type = "mesh", path = "{mesh}" }}
transforms = [ {{ rotate_y = 0.7 }} ]
[[objects]]
brdf = {{ type = "diffuse", kd = [0.5, 0.5, 0.5] }}
geometry = {{ type = "plane", pos = [0.0, -3.0, 0.0], n = [0.0, 1.0, 0.0] }}
[[objects]]
emitted = [20.0, 20.0, 20.0]
brdf = {{ type = "diffuse", kd = [0.0, 0.0, 0.0] }}
geometry = {{ type = "sphere", pos = [3.0, 8.0, 3.0], r = 1.0 }}
"""
    g = rtb.Scene.from_toml_string(text, assets_dir=ASSETS)
    o = oracle_mod.OracleScene.from_toml_string(text, ASSETS)
    assert g.info.n_triangles == n_tri
    tris = o.mesh_triangles(0).reshape(-1, 3)
    c, ext = tris.mean(0), (tris.max(0) - tris.min(0)).max()
    rng = np.random.default_rng(2)
    n = 100_000
    org = (c + rng.normal(size=(n, 3)) * ext).astype(np.float32)
    tgt = c + rng.uniform(-0.5, 0.5, size=(n, 3)) * ext
    d = tgt - org
    d = (d / np.linalg.norm(d, axis=1, keepdims=True)).astype(np.float32)
    d /= np.linalg.norm(d.astype(np.float64), axis=1, keepdims=True).astype(np.float32)
    ro = o.trace_rays(org.astype(np.float64), d.astype(np.float64))
    rg = g.trace_rays(org, d, count_work=True)
    mism = (ro["obj"] != rg["obj"]) | (ro["tri"] != rg["tri"])
    assert (ro["obj"] == 0).mean() > 0.2
    assert mism.mean() < 2e-3
    idx = np.flatnonzero(mism)
    if idx.size:
        amb = ambiguous_mask(o, org[idx].astype(np.float64), d[idx].astype(np.float64), {k: v[idx] for k, v in ro.items()}, rg["t"][idx])
        assert (~amb).mean() < 0.1
    assert rg["work"]["node_visits"] > 0 and rg["work"]["tri_tests"] > 0


# every scene at the reference server's frame size, and the BVH-heavy scene at the two sizes BASELINE.json's
# configs[2] / configs[3] are quoted on (camera rays, pixel counters and accumulator indices all depend on the size)
PATH_CASES = [(n, 600, 450, 64) for n in SCENE_NAMES] + [("flying_unicorn", 1920, 1080, 256), ("flying_unicorn", 3840, 2160, 4096),
                                                         ("cubes", 3840, 2160, 4096)]


@pytest.mark.parametrize("name,W,H,spp", PATH_CASES, ids=[f"{n}-{w}x{h}" for n, w, h, _ in PATH_CASES])
@pytest.mark.parametrize("use_mis", [False, True])
def test_path_radiance_same_random_numbers(gpu_scene, oracle_scene, oracle_mod, parity_log, name, W, H, spp, use_mis):
    # Both sides draw identical Philox numbers (RNG contract), so individual camera paths agree to fp32
    # accuracy except where a discrete decision (silhouette, roulette threshold) flips.
    g, o = gpu_scene(name), oracle_scene(name)
    o.set_modes(oracle_mod.ACCEL_EXACT, oracle_mod.EST_MIS_DEAD if use_mis else oracle_mod.EST_NEE)
    n = 20000
    rng = np.random.default_rng(11)
    px, py, si = rng.integers(0, W, n), rng.integers(0, H, n), rng.integers(0, spp, n)
    Lo = o.sample_radiance(W, H, spp, 42, px, py, si)
    Lg = g.sample_radiance(W, H, spp, px, py, si, seed=42, use_mis=use_mis).astype(np.float64)
    o.set_modes(oracle_mod.ACCEL_EXACT, oracle_mod.EST_NEE)
    fin = np.isfinite(Lo).all(axis=1) & np.isfinite(Lg).all(axis=1)
    assert fin.mean() > 0.999
    err = path_error(Lg[fin], Lo[fin])
    parity_log(f"gpu/path_radiance/{name}/{W}x{H}/{'mis_dead' if use_mis else 'nee'}", paths=n, finite=fin.mean(),
               err_median=np.median(err), err_q90=np.quantile(err, 0.9), err_q99=np.quantile(err, 0.99),
               frac_beyond_1e3=(err > 1e-3).mean(), mean_gpu=Lg[fin].mean(), mean_oracle=Lo[fin].mean())
    assert np.median(err) < 1e-5
    assert (err > 1e-3).mean() < (0.05 if use_mis else 0.02)
    if not use_mis:   # the dead branch is heavy-tailed (negative / huge weights): means are not comparable at n = 20000
        assert Lg[fin].mean() == pytest.approx(Lo[fin].mean(), rel=0.01)


mre = channel_mre   # relative error of the channel means (the weak form; pixel_mre gates beside it)


@pytest.mark.parametrize("name", SCENE_NAMES)
@pytest.mark.parametrize("use_mis", [False, True])
def test_frame_matches_oracle_same_seed(gpu_scene, oracle_scene, oracle_mod, parity_log, name, use_mis):
    g, o = gpu_scene(name), oracle_scene(name)
    o.set_modes(oracle_mod.ACCEL_EXACT, oracle_mod.EST_MIS_DEAD if use_mis else oracle_mod.EST_NEE)
    W, H, spp = 120, 90, 64
    io = o.render(W, H, spp, seed=3, nthreads=-NCPU)["rgb8"]
    o.set_modes(oracle_mod.ACCEL_EXACT, oracle_mod.EST_NEE)
    ig = g.render(W, H, spp, seed=3, use_mis=use_mis)
    d = np.abs(ig.astype(int) - io.astype(int))
    parity_log(f"gpu/frame_same_seed/{name}/{'mis_dead' if use_mis else 'nee'}", size=[W, H], spp=spp, pixel_mre=pixel_mre(ig, io, blur=1),
               pixel_mre_blur5=pixel_mre(ig, io), channel_mre=mre(ig, io), psnr=psnr(ig, io), frac_beyond_2_levels=(d > 2).mean(), max_level_diff=int(d.max()))
    assert (pixel_mre(ig, io, blur=1) < 0.01).all()       # <= 1 % mean relative error per channel, pixel by pixel
    assert (mre(ig, io) < 0.01).all()
    assert psnr(ig, io) >= 40.0
    assert (d > 2).mean() < (0.03 if use_mis else 0.005)
    st = g.stats()
    assert st["samples"] == W * H * spp


@pytest.mark.parametrize("W,H", [(1920, 1080), (3840, 2160)])
def test_rows_of_the_bench_frames_match_oracle(gpu_scene, oracle_scene, parity_log, W, H):
    # BASELINE.json configs[2] / configs[3] sizes: the oracle renders a few scan lines of the full-size frame (through the
    # Pegasus, its mirror image and the light), the GPU the whole frame with the same seed — the bytes of those rows must agree
    g, o = gpu_scene("flying_unicorn"), oracle_scene("flying_unicorn")
    spp, seed = 16, 31
    y0, stride = int(H * 0.07), H // 14
    rows = list(range(y0, H, stride))                      # 14 scan lines, one oracle call (rows are scheduled over the host threads)
    want = o.render(W, H, spp, seed=seed, y0=y0, y1=H, row_stride=stride, nthreads=-NCPU)["rgb8"][rows]
    got = g.render(W, H, spp, seed=seed)[rows]
    d = np.abs(got.astype(int) - want.astype(int))
    parity_log(f"gpu/bench_frame_rows/flying_unicorn/{W}x{H}", rows=rows, spp=spp, pixel_mre=pixel_mre(got, want, blur=1), psnr=psnr(got, want),
               frac_beyond_2_levels=(d > 2).mean(), max_level_diff=int(d.max()))
    assert (pixel_mre(got, want, blur=1) < 0.01).all() and psnr(got, want) >= 40.0
    assert (d > 2).mean() < 0.01


def test_converged_frame_independent_seeds(gpu_scene, oracle_scene, parity_log):
    # statistical form of the 1 % / 40 dB gate: oracle and GPU with DIFFERENT seeds, against the noise floor
    # of two oracle renders.  Small frame, 1024 spp (the oracle is a scalar CPU program).
    g, o = gpu_scene("cornell_box"), oracle_scene("cornell_box")
    W, H, spp = 64, 48, 1024
    a = o.render(W, H, spp, seed=100, nthreads=-NCPU)["rgb8"]
    b = o.render(W, H, spp, seed=200, nthreads=-NCPU)["rgb8"]
    c = g.render(W, H, spp, seed=300)
    floor = psnr(a, b)
    parity_log("gpu/frame_independent_seeds/cornell_box", size=[W, H], spp=spp, psnr_gpu_vs_oracle=psnr(c, a), psnr_oracle_vs_oracle=floor,
               pixel_mre_blur5=pixel_mre(c, a), pixel_mre_blur5_oracle_vs_oracle=pixel_mre(b, a), channel_mre=mre(c, a))
    assert (mre(c, a) < 0.01).all()
    assert (pixel_mre(c, a) < 1.3 * pixel_mre(b, a) + 1e-3).all()
    assert psnr(c, a) >= min(40.0, floor - 1.0)
    assert psnr(c, a) >= floor - 1.5                      # indistinguishable from a third oracle render


def test_direct_light_closed_form_gpu(rtb):
    # same closed form as tests/test_oracle_pins.py::test_direct_light_closed_form: L = kd Le (r/d)^2
    kd, Le, r, d = 0.5, 10.0, 1.0, 10.0
    text = f"""
[camera]
pos = [0.0, 5.0, 20.0]
dir = [0.0, -0.25, -1.0]
[[objects]]
brdf = {{ type = "diffuse", kd = [{kd}, {kd}, {kd}] }}
geometry = {{ type = "plane", pos = [0.0, 0.0, 0.0], n = [0.0, 1.0, 0.0] }}
[[objects]]
emitted = [{Le}, {Le}, {Le}]
brdf = {{ type = "diffuse", kd = [0.0, 0.0, 0.0] }}
geometry = {{ type = "sphere", pos = [0.0, {d}, 0.0], r = {r} }}
"""
    g = rtb.Scene.from_toml_string(text)
    n = 40000
    L = g.sample_radiance(101, 101, 4 * n, np.full(n, 50), np.full(n, 50), np.arange(n), seed=5)
    assert L.mean(axis=0) == pytest.approx([kd * Le * (r / d) ** 2] * 3, rel=0.01)


PHONG_SCENE = """
[camera]
pos = [50.0, 52.0, 295.6]
dir = [0.0, -0.042612, -1.0]
[[objects]]
brdf = { type = "diffuse", kd = [0.75, 0.25, 0.25] }
geometry = { type = "plane", pos = [1.0, 0.0, 0.0], n = [-1.0, 0.0, 0.0] }
[[objects]]
brdf = { type = "diffuse", kd = [0.25, 0.25, 0.75] }
geometry = { type = "plane", pos = [99.0, 0.0, 0.0], n = [-1.0, 0.0, 0.0] }
[[objects]]
brdf = { type = "phong", kd = 0.5, ks = 0.4, power = 8, color_d = [0.8, 0.8, 0.3], color_s = [1.0, 1.0, 1.0] }
geometry = { type = "plane", pos = [0.0, 0.0, 0.0], n = [0.0, 1.0, 0.0] }
[[objects]]
brdf = { type = "diffuse", kd = [0.75, 0.75, 0.75] }
geometry = { type = "plane", pos = [0.0, 0.0, 0.0], n = [0.0, 0.0, -1.0] }
[[objects]]
brdf = { type = "specular", ks = [0.9, 0.9, 0.9] }
geometry = { type = "sphere", pos = [30.0, 16.5, 60.0], r = 16.5 }
[[objects]]
brdf = { type = "specular", ks = [0.9, 0.8, 0.7] }
geometry = { type = "sphere", pos = [70.0, 16.5, 90.0], r = 16.5 }
[[objects]]
brdf = { type = "phong", kd = 0.2, ks = 0.7, power = 30, color_d = [0.3, 0.9, 0.3], color_s = [1.0, 1.0, 1.0] }
geometry = { type = "cube", pos = [40.0, 0.0, 120.0], size = 14.0 }
transforms = [ { rotate_y = 0.4 } ]
[[objects]]
emitted = [40.0, 40.0, 40.0]
brdf = { type = "diffuse", kd = [0.0, 0.0, 0.0] }
geometry = { type = "sphere", pos = [50.0, 70.0, 100.0], r = 5.0 }
"""


def test_phong_and_specular_chains(rtb, oracle_mod):
    # Phong (local-frame sampling quirk, src/scene.rs:69-96) and mirror->mirror chains where the reference
    # hands the stale `o` down the recursion (src/scene.rs:178); no reference scene exercises either
    g = rtb.Scene.from_toml_string(PHONG_SCENE)
    o = oracle_mod.OracleScene.from_toml_string(PHONG_SCENE)
    W, H, spp, n = 200, 150, 32, 20000
    rng = np.random.default_rng(4)
    px, py, si = rng.integers(0, W, n), rng.integers(0, H, n), rng.integers(0, spp, n)
    Lo = o.sample_radiance(W, H, spp, 9, px, py, si)
    Lg = g.sample_radiance(W, H, spp, px, py, si, seed=9).astype(np.float64)
    fin = np.isfinite(Lo).all(axis=1) & np.isfinite(Lg).all(axis=1)
    assert fin.mean() > 0.99
    err = np.abs(Lg[fin] - Lo[fin]).max(axis=1) / (np.abs(Lo[fin]).max(axis=1) + 1e-3)
    assert np.median(err) < 2e-5 and (err > 1e-3).mean() < 0.03
    io = o.render(80, 60, 32, seed=1, nthreads=-NCPU)["rgb8"]
    ig = g.render(80, 60, 32, seed=1)
    assert psnr(ig, io) >= 38.0 and (mre(ig, io) < 0.015).all()


MESH_LIGHT = """
[camera]
pos = [0.0, 3.0, 12.0]
dir = [0.0, -0.2, -1.0]
[[objects]]
brdf = { type = "diffuse", kd = [0.6, 0.6, 0.6] }
geometry = { type = "plane", pos = [0.0, 0.0, 0.0], n = [0.0, 1.0, 0.0] }
[[objects]]
emitted = [8.0, 6.0, 4.0]
brdf = { type = "diffuse", kd = [0.0, 0.0, 0.0] }
geometry = { type = "prism", pos = [-1.0, 4.0, -1.0], size = [2.0, 0.5, 2.0] }
[[objects]]
brdf = { type = "diffuse", kd = [0.4, 0.7, 0.4] }
geometry = { type = "sphere", pos = [2.0, 1.0, 0.0], r = 1.0 }
"""


def test_mesh_light_sampling_quirk(rtb, oracle_mod):
    # Geometry::sample for a mesh (src/geometry.rs:588-592): area-weighted triangle, then
    # Triangle::get_barycentric WITHOUT the `+ a` (src/geometry.rs:622-628) — reproduced, not fixed
    g = rtb.Scene.from_toml_string(MESH_LIGHT)
    o = oracle_mod.OracleScene.from_toml_string(MESH_LIGHT)
    assert g.light_source == o.light_source == 1
    W, H, spp, n = 120, 90, 16, 8000
    rng = np.random.default_rng(8)
    px, py, si = rng.integers(0, W, n), rng.integers(0, H, n), rng.integers(0, spp, n)
    Lo = o.sample_radiance(W, H, spp, 2, px, py, si)
    Lg = g.sample_radiance(W, H, spp, px, py, si, seed=2).astype(np.float64)
    fin = np.isfinite(Lo).all(axis=1) & np.isfinite(Lg).all(axis=1)
    err = np.abs(Lg[fin] - Lo[fin]).max(axis=1) / (np.abs(Lo[fin]).max(axis=1) + 1e-3)
    assert fin.mean() > 0.99 and np.median(err) < 2e-5 and (err > 1e-3).mean() < 0.03


def test_mesh_only_scene_and_tiny_meshes(rtb, oracle_mod, tmp_path):
    # no analytic surface except the light: rays can miss everything (received_radiance returns 0, src/scene.rs:156-158);
    # a 2-triangle mesh is a single LBVH leaf (no inner node at all), the prism a small tree
    (tmp_path / "quad.obj").write_text("v -6 0 -6\nv 6 0 -6\nv 6 0 6\nv -6 0 6\nf 1 2 3\nf 1 3 4\n")
    text = """
[camera]
pos = [0.0, 6.0, 14.0]
dir = [0.0, -0.35, -1.0]
[[objects]]
brdf = { type = "diffuse", kd = [0.7, 0.6, 0.5] }
geometry = { type = "mesh", path = "quad.obj" }
[[objects]]
brdf = { type = "diffuse", kd = [0.3, 0.8, 0.3] }
geometry = { type = "prism", pos = [-1.0, 0.0, -1.0], size = [2.0, 3.0, 2.0] }
transforms = [ { rotate_y = 0.5 } ]
[[objects]]
emitted = [30.0, 30.0, 30.0]
brdf = { type = "diffuse", kd = [0.0, 0.0, 0.0] }
geometry = { type = "sphere", pos = [3.0, 7.0, 2.0], r = 1.0 }
"""
    g = rtb.Scene.from_toml_string(text, assets_dir=str(tmp_path))
    o = oracle_mod.OracleScene.from_toml_string(text, str(tmp_path))
    assert g.info.n_planes == 0 and g.info.n_triangles == 14
    W, H = 160, 120
    org, dirs = o.primary_rays(W, H)
    ro, rg = o.trace_rays(org, dirs), g.trace_primary(W, H)
    mism = (ro["obj"] != rg["obj"]) | (ro["tri"] != rg["tri"])
    assert (ro["obj"] < 0).mean() > 0.2 and (ro["obj"] == 0).any() and (ro["obj"] == 1).any()
    if mism.any():
        idx = np.flatnonzero(mism)
        assert ambiguous_mask(o, org[idx], dirs[idx], {k: v[idx] for k, v in ro.items()}, rg["t"][idx]).all()
    assert mism.mean() < 1e-3
    n, spp = 6000, 16
    rng = np.random.default_rng(3)
    px, py, si = rng.integers(0, W, n), rng.integers(0, H, n), rng.integers(0, spp, n)
    Lo = o.sample_radiance(W, H, spp, 5, px, py, si)
    Lg = g.sample_radiance(W, H, spp, px, py, si, seed=5).astype(np.float64)
    err = np.abs(Lg - Lo).max(axis=1) / (np.abs(Lo).max(axis=1) + 1e-3)
    assert np.median(err) < 1e-5 and (err > 1e-3).mean() < 0.02
    io = o.render(80, 60, 32, seed=2, nthreads=-NCPU)["rgb8"]
    ig = g.render(80, 60, 32, seed=2)
    assert psnr(ig, io) >= 40.0


def test_random_triangle_soup_lbvh(rtb, oracle_mod, tmp_path):
    # LBVH stress: an unstructured soup (overlapping boxes, slivers, wildly different sizes, duplicated centroids)
    # handed over through rtb_scene_create; the oracle reads the same triangles from an OBJ file
    rng = np.random.default_rng(12)
    n = 3000
    centres = rng.uniform(-10, 10, size=(n, 1, 3))
    centres[:200] = centres[0]                       # 200 triangles share one centroid cell (equal Morton codes)
    size = np.exp(rng.uniform(np.log(0.02), np.log(6.0), size=(n, 1, 1)))
    tris = (centres + rng.normal(size=(n, 3, 3)) * size).astype(np.float32)
    with open(tmp_path / "soup.obj", "w") as f:
        for t in tris.reshape(-1, 3):
            f.write(f"v {float(t[0])!r} {float(t[1])!r} {float(t[2])!r}\n")
        for i in range(n):
            f.write(f"f {3 * i + 1} {3 * i + 2} {3 * i + 3}\n")
    text = """
[camera]
pos = [0.0, 0.0, 40.0]
dir = [0.0, 0.0, -1.0]
[[objects]]
brdf = { type = "diffuse", kd = [0.7, 0.7, 0.7] }
geometry = { type = "mesh", path = "soup.obj" }
[[objects]]
emitted = [20.0, 20.0, 20.0]
brdf = { type = "diffuse", kd = [0.0, 0.0, 0.0] }
geometry = { type = "sphere", pos = [0.0, 30.0, 0.0], r = 2.0 }
"""
    o = oracle_mod.OracleScene.from_toml_string(text, str(tmp_path))
    g = rtb.Scene.from_objects((0, 0, 40), (0, 0, -1), [
        {"brdf": ("diffuse", (0.7, 0.7, 0.7)), "geometry": ("mesh", tris)},
        {"emitted": (20, 20, 20), "brdf": ("diffuse", (0, 0, 0)), "geometry": ("sphere", (0, 30, 0), 2.0)}])
    assert g.info.n_triangles == n and np.array_equal(g.triangles(), o.mesh_triangles(0).astype(np.float32))
    m = 150_000
    org = rng.uniform(-25, 25, size=(m, 3)).astype(np.float32)
    d = rng.normal(size=(m, 3))
    d = (d / np.linalg.norm(d, axis=1, keepdims=True)).astype(np.float32)
    d /= np.linalg.norm(d.astype(np.float64), axis=1, keepdims=True).astype(np.float32)
    ro = o.trace_rays(org.astype(np.float64), d.astype(np.float64))
    rg = g.trace_rays(org, d)
    assert (ro["obj"] == 0).mean() > 0.2
    mism = (ro["obj"] != rg["obj"]) | (ro["tri"] != rg["tri"])
    assert mism.mean() < 3e-3
    idx = np.flatnonzero(mism)
    if idx.size:
        amb = ambiguous_mask(o, org[idx].astype(np.float64), d[idx].astype(np.float64), {k: v[idx] for k, v in ro.items()}, rg["t"][idx])
        assert (~amb).sum() <= max(3, 0.05 * idx.size)
    ok = ~mism & (ro["obj"] >= 0)
    rel = np.abs(rg["t"][ok].astype(np.float64) - ro["t"][ok]) / np.maximum(ro["t"][ok], 1e-2)
    assert np.quantile(rel, 0.999) < T_REL_TOL


@pytest.mark.gpu
def test_every_hierarchy_builder_gives_the_same_hits(rtb, gpu_scene, monkeypatch):
    # RTB_BVH picks the hierarchy over the same triangles: binned SAH (default, top-down on the device), PLOC, Karras, and the
    # host-side SAH the device builder was checked against.  Nearest hits do not depend on the tree; the SAH tree is the shallowest.
    g0 = gpu_scene("flying_unicorn")
    rng = np.random.default_rng(9)
    n = 100_000
    lo, hi = np.array(g0.info.bvh_min), np.array(g0.info.bvh_max)
    org = (lo + (hi - lo) * rng.random((n, 3)) * 1.6 - 0.3 * (hi - lo)).astype(np.float32)
    d = rng.normal(size=(n, 3))
    d = (d / np.linalg.norm(d, axis=1, keepdims=True)).astype(np.float32)
    a = g0.trace_rays(org, d)
    assert (a["tri"] >= 0).mean() > 0.05
    f0 = g0.render(160, 120, 16, seed=2).astype(int)
    info = {"sah": (g0.info.bvh_nodes, g0.info.bvh_depth)}
    for mode in ("ploc", "lbvh", "sah_host"):
        monkeypatch.setenv("RTB_BVH", mode)
        g = rtb.Scene.from_toml(scene_path("flying_unicorn"), device=0)
        monkeypatch.delenv("RTB_BVH")
        b = g.trace_rays(org, d)
        assert np.array_equal(a["obj"], b["obj"]) and np.array_equal(a["t"], b["t"]), mode
        assert (a["tri"] != b["tri"]).mean() < 1e-4, mode      # exact distance ties on shared edges only
        assert np.abs(f0 - g.render(160, 120, 16, seed=2).astype(int)).max() <= 1, mode
        info[mode] = (g.info.bvh_nodes, g.info.bvh_depth)
    assert info["sah"][1] <= min(info["ploc"][1], info["lbvh"][1])
    assert abs(info["sah"][0] - info["sah_host"][0]) <= 0.02 * info["sah"][0]    # same policy, same tree up to float rounding of the bins
    # the build is deterministic: integer atomics and scans only
    g1 = rtb.Scene.from_toml(scene_path("flying_unicorn"), device=0)
    e0, e1 = g0.export(), g1.export()
    e0[152:160] = e1[152:160] = 0            # ExportHeader.build_ms, the one field that is a measurement
    assert np.array_equal(e0, e1)


@pytest.mark.gpu
def test_sah_builder_splits_coinciding_centroids(rtb):
    # 40 copies of one triangle (no centroid extent: no bin can separate them -> halved by triangle index until 8 fit a leaf)
    # next to 200 distinct ones; every builder must still find the same nearest hit
    rng = np.random.default_rng(4)
    base = np.array([[0, 0, 0], [4, 0, 0], [0, 4, 0]], dtype=np.float64)
    tris = [base.copy() for _ in range(40)]
    for _ in range(200):
        c = rng.uniform(-20, 20, 3)
        tris.append(c + rng.normal(size=(3, 3)) * 2.0)
    tris = np.array(tris)
    objs = [{"brdf": ("diffuse", (0.7, 0.7, 0.7)), "geometry": ("mesh", tris)},
            {"emitted": (20, 20, 20), "brdf": ("diffuse", (0, 0, 0)), "geometry": ("sphere", (0, 60, 0), 2.0)}]
    g = rtb.Scene.from_objects((0, 0, 60), (0, 0, -1), objs)
    os.environ["RTB_BVH"] = "lbvh"
    try:
        k = rtb.Scene.from_objects((0, 0, 60), (0, 0, -1), objs)
    finally:
        del os.environ["RTB_BVH"]
    m = 50_000
    org = rng.uniform(-30, 30, size=(m, 3)).astype(np.float32)
    d = rng.normal(size=(m, 3))
    d = (d / np.linalg.norm(d, axis=1, keepdims=True)).astype(np.float32)
    a, b = g.trace_rays(org, d), k.trace_rays(org, d)
    assert np.array_equal(a["obj"], b["obj"]) and np.array_equal(a["t"], b["t"])
    # straight down onto the stack of copies: the hit is one of them (the lowest index wins ties inside a leaf, any of the 40 across leaves)
    hit = g.trace_rays(np.array([[1, 1, 10]], np.float32), np.array([[0, 0, -1]], np.float32))
    assert hit["obj"][0] == 0 and 0 <= hit["tri"][0] < 40 and abs(hit["t"][0] - 10) < 1e-4


# ---------------------------------------------------------------- ACCEL_OCTREE_REFERENCE: the reference's real mesh path
@pytest.mark.parametrize("name", ["cubes", "flying_unicorn"])
def test_octree_mode_returns_the_reference_hits(rtb, gpu_scene, oracle_scene, oracle_mod, parity_log, name):
    # Octree::intersect is not a nearest-hit query (early exit on the first child with any hit, src/geometry.rs:1263-1273);
    # the device traversal must return the SAME (possibly non-nearest) triangle as the oracle's octree_faithful mode
    g, o = gpu_scene(name), oracle_scene(name)
    W, H = 600, 450
    org, dirs = o.primary_rays(W, H, 0, 0, 0.0, 0.0)
    rng = np.random.default_rng(9)
    n = 200_000
    lo, hi = np.array(g.info.bvh_min, dtype=np.float64), np.array(g.info.bvh_max, dtype=np.float64)
    so = lo + (hi - lo) * (rng.random((n, 3)) * 1.4 - 0.2)          # origins in and around the meshes: the secondary-ray case
    sd = rng.normal(size=(n, 3))
    sd /= np.linalg.norm(sd, axis=1, keepdims=True)
    org32 = np.concatenate([org, so]).astype(np.float32)
    d32 = np.concatenate([dirs, sd]).astype(np.float32)
    d32 /= np.linalg.norm(d32.astype(np.float64), axis=1, keepdims=True).astype(np.float32)
    o.set_modes(oracle_mod.ACCEL_OCTREE_FAITHFUL, oracle_mod.EST_NEE)
    ro = o.trace_rays(org32.astype(np.float64), d32.astype(np.float64))
    o.set_modes(oracle_mod.ACCEL_EXACT, oracle_mod.EST_NEE)
    rx = o.trace_rays(org32.astype(np.float64), d32.astype(np.float64))
    rg = g.trace_rays(org32, d32, accel=rtb.ACCEL_OCTREE_REFERENCE)
    differ = (ro["obj"] != rg["obj"]) | (ro["tri"] != rg["tri"])
    # two surfaces at the same distance (the cubes' bottom faces lie IN the floor plane, two triangles share an edge): which one
    # is reported is decided by rounding on both sides — the same exclusion as ambiguous_mask's first rule
    with np.errstate(invalid="ignore"):
        tie = differ & (np.abs(rg["t"].astype(np.float64) - ro["t"]) <= 1e-5 * np.abs(ro["t"]))
    mism = differ & ~tie
    non_nearest = (ro["tri"] != rx["tri"]) | (ro["obj"] != rx["obj"])      # where the reference itself misses the nearest triangle
    ok = ~differ & (ro["obj"] >= 0)
    rel = np.abs(rg["t"][ok].astype(np.float64) - ro["t"][ok]) / np.maximum(ro["t"][ok], 1e-3)
    parity_log(f"gpu/octree_mode_rays/{name}", rays=int(mism.size), mesh_hits=int((ro["tri"] >= 0).sum()), mismatches=int(mism.sum()), equal_distance_ties=int(tie.sum()),
               reference_non_nearest_hits=int(non_nearest.sum()), gpu_agrees_on_those=int((non_nearest & ~mism).sum()),
               t_rel_q9999=np.quantile(rel, 0.9999))
    assert mism.mean() < 1e-3            # fp32 vs f64 decisions at box faces / triangle edges
    assert np.quantile(rel, 0.9999) < T_REL_TOL
    if name == "flying_unicorn":
        assert non_nearest.sum() > 1000 and (non_nearest & ~mism).sum() > 0.98 * non_nearest.sum()   # the defect itself is reproduced


@pytest.mark.parametrize("name", ["cubes", "flying_unicorn"])
def test_octree_mode_path_radiance(rtb, gpu_scene, oracle_scene, oracle_mod, parity_log, name):
    g, o = gpu_scene(name), oracle_scene(name)
    W, H, spp, n = 600, 450, 64, 20000
    rng = np.random.default_rng(13)
    px, py, si = rng.integers(0, W, n), rng.integers(0, H, n), rng.integers(0, spp, n)
    o.set_modes(oracle_mod.ACCEL_OCTREE_FAITHFUL, oracle_mod.EST_NEE)
    Lo = o.sample_radiance(W, H, spp, 42, px, py, si)
    o.set_modes(oracle_mod.ACCEL_EXACT, oracle_mod.EST_NEE)
    Lg = g.sample_radiance(W, H, spp, px, py, si, seed=42, accel=rtb.ACCEL_OCTREE_REFERENCE).astype(np.float64)
    fin = np.isfinite(Lo).all(axis=1) & np.isfinite(Lg).all(axis=1)
    err = path_error(Lg[fin], Lo[fin])
    parity_log(f"gpu/octree_mode_path_radiance/{name}", paths=n, err_median=np.median(err), err_q99=np.quantile(err, 0.99), frac_beyond_1e3=(err > 1e-3).mean())
    assert fin.mean() > 0.999 and np.median(err) < 1e-5 and (err > 1e-3).mean() < 0.03
