"""Rough metal (brdf 4, k_shade MODE 6 / 7) on the GPU: per-path radiance against the f64 metal oracle under shared random
numbers, frames, the single-sphere-light identity of the all-lights estimator, the scheduling of the wavefront loop, the
refusal of the dead-MIS estimator, jobs, guides and export / import."""
import numpy as np
import pytest

from conftest import NCPU
from parity_metrics import path_error, psnr

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def metal(oracle_mod):
    """the f64 oracle with metal (tests/metal_oracle.py); oracle_mod builds the oracle whose entry points it shares"""
    import metal_oracle

    metal_oracle.lib()
    return metal_oracle


# smallpt's box with a near-polished metal floor, a rough gold sphere, a rotated aluminium cube (a mesh), a mirror that sees
# the metals (mirror -> metal chains: the metal must use the true direction of arrival), a glass sphere and one sphere light;
# SECOND_LIGHT adds another one for the all-lights estimator
METAL_SCENE = """
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
brdf = { type = "diffuse", kd = [0.75, 0.75, 0.75] }
geometry = { type = "plane", pos = [0.0, 0.0, 0.0], n = [0.0, 0.0, -1.0] }
[[objects]]
brdf = { type = "metal", roughness = 0.08, color = [0.95, 0.93, 0.88] }
geometry = { type = "plane", pos = [0.0, 0.0, 0.0], n = [0.0, 1.0, 0.0] }
[[objects]]
brdf = { type = "diffuse", kd = [0.75, 0.75, 0.75] }
geometry = { type = "plane", pos = [0.0, 81.6, 0.0], n = [0.0, -1.0, 0.0] }
[[objects]]
brdf = { type = "specular", ks = [0.9, 0.9, 0.9] }
geometry = { type = "sphere", pos = [20.0, 12.0, 40.0], r = 12.0 }
[[objects]]
brdf = { type = "metal", roughness = 0.3, color = [1.0, 0.71, 0.29] }
geometry = { type = "sphere", pos = [73.0, 16.5, 78.0], r = 16.5 }
[[objects]]
brdf = { type = "dielectric", ior = 1.5 }
geometry = { type = "sphere", pos = [30.0, 9.0, 100.0], r = 9.0 }
[[objects]]
brdf = { type = "metal", roughness = 0.6, color = [0.91, 0.92, 0.92] }
geometry = { type = "cube", pos = [42.0, 0.0, 60.0], size = 16.0 }
transforms = [ { rotate_y = 0.5 } ]
[[objects]]
emitted = [40.0, 40.0, 40.0]
brdf = { type = "diffuse", kd = [0.0, 0.0, 0.0] }
geometry = { type = "sphere", pos = [50.0, 70.0, 100.0], r = 5.0 }
"""
SECOND_LIGHT = """
[[objects]]
emitted = [6.0, 12.0, 30.0]
brdf = { type = "diffuse", kd = [0.0, 0.0, 0.0] }
geometry = { type = "sphere", pos = [20.0, 60.0, 60.0], r = 6.0 }
"""
TWO_LIGHTS = METAL_SCENE + SECOND_LIGHT
RAY_KEYS = ("samples", "rays_primary", "rays_extension", "rays_shadow", "rays_bvh", "shadow_bvh")


@pytest.fixture(scope="module")
def scenes(rtb, metal):
    return {"one": rtb.Scene.from_toml_string(METAL_SCENE), "two": rtb.Scene.from_toml_string(TWO_LIGHTS)}


@pytest.mark.parametrize("estimator, octree", [(0, False), (3, False), (0, True), (3, True)])
def test_path_radiance_matches_the_oracle(rtb, metal, scenes, parity_log, estimator, octree):
    g = scenes["two"]
    o = metal.OracleScene.from_toml_string(TWO_LIGHTS)
    W, H, spp, n = 200, 150, 32, 20000
    rng = np.random.default_rng(41 + estimator)
    px, py, si = rng.integers(0, W, n), rng.integers(0, H, n), rng.integers(0, spp, n)
    o.set_modes(metal.ACCEL_OCTREE_FAITHFUL if octree else metal.ACCEL_EXACT, estimator)
    Lo = o.sample_radiance(W, H, spp, 9, px, py, si)
    Lg = g.sample_radiance(W, H, spp, px, py, si, seed=9, estimator=estimator,
                           accel=rtb.ACCEL_OCTREE_REFERENCE if octree else 0).astype(np.float64)
    fin = np.isfinite(Lo).all(axis=1) & np.isfinite(Lg).all(axis=1)
    err = path_error(Lg[fin], Lo[fin])
    parity_log(f"gpu/metal/path_radiance/est{estimator}{'_octree' if octree else ''}", paths=n, err_median=np.median(err),
               frac_beyond_1e3=(err > 1e-3).mean(), mean_gpu=Lg[fin].mean(0), mean_oracle=Lo[fin].mean(0))
    assert fin.mean() > 0.99 and Lo[fin].sum() > 0
    assert np.median(err) < 2e-5 and (err > 1e-3).mean() < 0.03


def test_frame_matches_the_oracle(metal, scenes, parity_log):
    g = scenes["one"]
    o = metal.OracleScene.from_toml_string(METAL_SCENE)
    io = o.render(80, 60, 32, seed=1, nthreads=-NCPU)["rgb8"]
    ig = g.render(80, 60, 32, seed=1)
    a, b = ig.reshape(-1, 3).astype(np.float64), io.reshape(-1, 3).astype(np.float64)
    mre = np.abs(a.mean(0) - b.mean(0)) / b.mean(0)
    parity_log("gpu/metal/frame", psnr=psnr(ig, io), mre=mre)
    assert psnr(ig, io) >= 38.0 and (mre < 0.015).all()


def test_single_sphere_light_equals_nee(rtb, scenes, parity_log):
    g = scenes["one"]
    W, H, spp, n = 600, 450, 64, 100000
    rng = np.random.default_rng(5)
    px, py, si = rng.integers(0, W, n), rng.integers(0, H, n), rng.integers(0, spp, n)
    nee = g.sample_radiance(W, H, spp, px, py, si, seed=4).astype(np.float64)
    alll = g.sample_radiance(W, H, spp, px, py, si, seed=4, estimator=rtb.EST_NEE_ALL_LIGHTS).astype(np.float64)
    d = np.abs(alll - nee).max(axis=1)
    parity_log("gpu/metal/single_light", paths=n, median=np.median(d), frac_within_1e4=(d <= 1e-4).mean())
    assert nee.sum() > 0
    assert np.median(d) < 1e-6 and (d <= 1e-4).mean() >= 0.999


@pytest.mark.parametrize("estimator", [0, 3])
def test_scheduling_does_not_change_the_frame(rtb, scenes, monkeypatch, estimator):
    g = scenes["two"]
    W, H, spp = 200, 150, 64
    ref = g.render(W, H, spp, seed=17, estimator=estimator).astype(int)
    base = g.stats()
    assert base["rays_extension"] > 0
    for env in ("RTB_NO_FAST_SHADE", "RTB_NO_SMALL_TABLE", "RTB_GENERIC_TABLE"):
        monkeypatch.setenv(env, "1")
        f = g.render(W, H, spp, seed=17, estimator=estimator).astype(int)
        st = g.stats()
        monkeypatch.delenv(env)
        assert np.abs(f - ref).max() <= 1, env
        assert all(st[k] == base[k] for k in RAY_KEYS), (env, st, base)
    monkeypatch.setenv("RTB_INLINE_TAIL", "0")
    for kw in ({}, {"pool_paths": 1024}, {"pool_paths": 6000}):   # the inline tail off; two pool sizes
        f = g.render(W, H, spp, seed=17, estimator=estimator, **kw).astype(int)
        st = g.stats()
        assert np.abs(f - ref).max() <= 1, kw
        assert all(st[k] == base[k] for k in RAY_KEYS), (kw, st, base)   # the same rays, only their schedule differs
    monkeypatch.delenv("RTB_INLINE_TAIL")
    # two emulated ranks, untiled: the union of their tiles is the world = 1 frame
    out = np.zeros((H, W, 3), dtype=np.uint8)
    for r in range(2):
        g.render(W, H, spp, seed=17, rank=r, world=2, out=out, estimator=estimator)
    assert np.abs(out.astype(int) - ref).max() <= 1


def test_dead_mis_estimator_is_refused(rtb, scenes):
    g = scenes["one"]
    with pytest.raises(rtb.RtbError) as e:
        g.render(64, 48, 4, estimator=rtb.EST_MIS_DEAD)
    assert e.value.code == rtb.RTB_EUNSUPPORTED and "metal" in str(e.value)
    with pytest.raises(rtb.RtbError) as e:
        g.sample_radiance(64, 48, 4, [1], [1], [0], estimator=rtb.EST_MIS_DEAD)
    assert e.value.code == rtb.RTB_EUNSUPPORTED
    # the balance heuristic keeps plain next-event estimation at a metal vertex: same expectation
    assert abs(g.render(200, 150, 64, seed=3, estimator=rtb.EST_MIS_BALANCE).astype(float).mean() -
               g.render(200, 150, 64, seed=4).astype(float).mean()) < 0.02 * g.render(200, 150, 64, seed=4).mean()


def test_progressive_adaptive_and_denoised(rtb, scenes):
    g = scenes["two"]
    W, H, spp, seed = 200, 150, 64, 8
    for est in (rtb.EST_NEE, rtb.EST_NEE_ALL_LIGHTS):
        ref = g.render(W, H, spp, seed=seed, estimator=est).astype(int)
        job = rtb.RenderJob(g, W, H, spp, seed=seed, passes=4, estimator=est)
        frames = list(job.frames())
        assert not job.close() and len(frames) == 4
        assert np.abs(frames[-1][1].astype(int) - ref).max() <= 1
        job = rtb.RenderJob(g, W, H, spp, seed=seed, adaptive={"target_levels": 0.0, "pass_spp": 16}, estimator=est)
        frames = list(job.frames())
        assert not job.close()
        assert np.abs(frames[-1][1].astype(int) - ref).max() <= 1
        dn = g.render(W, H, spp, seed=seed, estimator=est, denoise=True)
        assert dn.shape == ref.shape and abs(dn.astype(float).mean() - ref.mean()) < 0.05 * ref.mean()


def test_guides_give_metal_its_f0(rtb):
    text = """
[camera]
pos = [0.0, 0.0, 10.0]
dir = [0.0, 0.0, -1.0]
[[objects]]
brdf = { type = "diffuse", kd = [0.5, 0.6, 0.7] }
geometry = { type = "plane", pos = [0.0, 0.0, -5.0], n = [0.0, 0.0, 1.0] }
[[objects]]
brdf = { type = "metal", roughness = 0.3, color = [1.0, 0.71, 0.29] }
geometry = { type = "sphere", pos = [0.0, 0.0, 0.0], r = 2.0 }
[[objects]]
emitted = [4.0, 4.0, 4.0]
brdf = { type = "diffuse", kd = [0.0, 0.0, 0.0] }
geometry = { type = "sphere", pos = [0.0, 8.0, 0.0], r = 1.0 }
"""
    g = rtb.Scene.from_toml_string(text)
    gb = g.gbuffer(65, 65)
    assert gb["obj"][32, 32] == 1
    assert np.allclose(gb["albedo"][32, 32], [1.0, 0.71, 0.29], rtol=1e-6)
    assert gb["depth"][32, 32] == pytest.approx(8.0, rel=1e-3)


def test_export_import_renders_the_same_frame(rtb, scenes):
    g = scenes["two"]
    again = rtb.Scene.from_export(g.export())
    for est in (rtb.EST_NEE, rtb.EST_NEE_ALL_LIGHTS):
        assert np.array_equal(again.render(200, 150, 32, seed=2, estimator=est), g.render(200, 150, 32, seed=2, estimator=est))
