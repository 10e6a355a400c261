"""The dielectric material (brdf 3) on the GPU: per-path radiance against the f64 oracle under shared random numbers,
frames, the closed-form transmittance of a glass sphere, every estimator, and the scheduling of the wavefront loop."""
import numpy as np
import pytest

from conftest import NCPU
from parity_metrics import path_error, psnr
from test_dielectric_cpu import AXIS_SCENE, AXIS_W, AXIS_WANT

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def glass(oracle_mod):
    """the f64 oracle with the dielectric (tests/glass_oracle.py); oracle_mod builds the oracle whose entry points it shares"""
    import glass_oracle

    glass_oracle.lib()
    return glass_oracle

# smallpt's box with a glass sphere, a tinted glass cube (a rotated mesh), a glass floor slab behind a plane (the medium is
# the half-space below it) and a mirror that sees the glass (mirror -> glass chains)
GLASS_SCENE = """
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
brdf = { type = "diffuse", kd = [0.75, 0.75, 0.75] }
geometry = { type = "plane", pos = [0.0, 0.0, 0.0], n = [0.0, 1.0, 0.0] }
[[objects]]
brdf = { type = "dielectric", ior = 1.33, tint = [0.8, 0.9, 1.0] }
geometry = { type = "plane", pos = [0.0, 4.0, 0.0], n = [0.0, 1.0, 0.0] }
[[objects]]
brdf = { type = "diffuse", kd = [0.75, 0.75, 0.75] }
geometry = { type = "plane", pos = [0.0, 81.6, 0.0], n = [0.0, -1.0, 0.0] }
[[objects]]
brdf = { type = "specular", ks = [0.9, 0.9, 0.9] }
geometry = { type = "sphere", pos = [27.0, 16.5, 47.0], r = 16.5 }
[[objects]]
brdf = { type = "dielectric", ior = 1.5 }
geometry = { type = "sphere", pos = [73.0, 16.5, 78.0], r = 16.5 }
[[objects]]
brdf = { type = "dielectric", ior = 1.6, tint = [0.9, 0.7, 0.5] }
geometry = { type = "cube", pos = [38.0, 4.0, 100.0], size = 14.0 }
transforms = [ { rotate_y = 0.5 }, { rotate_x = 0.2 } ]
[[objects]]
emitted = [40.0, 40.0, 40.0]
brdf = { type = "diffuse", kd = [0.0, 0.0, 0.0] }
geometry = { type = "sphere", pos = [50.0, 70.0, 100.0], r = 5.0 }
"""


@pytest.fixture(scope="module")
def scenes(rtb, glass):
    return rtb.Scene.from_toml_string(GLASS_SCENE), glass.OracleScene.from_toml_string(GLASS_SCENE)


@pytest.mark.parametrize("estimator, octree", [(0, False), (1, False), (0, True)])
def test_path_radiance_matches_the_oracle(rtb, glass, scenes, parity_log, estimator, octree):
    g, o = scenes
    W, H, spp, n = 200, 150, 32, 20000
    rng = np.random.default_rng(21 + estimator)
    px, py, si = rng.integers(0, W, n), rng.integers(0, H, n), rng.integers(0, spp, n)
    o.set_modes(glass.ACCEL_OCTREE_FAITHFUL if octree else glass.ACCEL_EXACT, estimator)
    Lo = o.sample_radiance(W, H, spp, 9, px, py, si)
    o.set_modes(glass.ACCEL_EXACT, glass.EST_NEE)
    Lg = g.sample_radiance(W, H, spp, px, py, si, seed=9, estimator=estimator,
                           accel=rtb.ACCEL_OCTREE_REFERENCE if octree else 0).astype(np.float64)
    fin = np.isfinite(Lo).all(axis=1) & np.isfinite(Lg).all(axis=1)
    err = path_error(Lg[fin], Lo[fin])
    parity_log(f"gpu/dielectric/path_radiance/est{estimator}{'_octree' if octree else ''}", paths=n, err_median=np.median(err),
               frac_beyond_1e3=(err > 1e-3).mean(), mean_gpu=Lg[fin].mean(0), mean_oracle=Lo[fin].mean(0))
    assert fin.mean() > 0.99
    assert np.median(err) < 2e-5 and (err > 1e-3).mean() < 0.03


def test_frame_matches_the_oracle(scenes, parity_log):
    g, o = scenes
    io = o.render(80, 60, 32, seed=1, nthreads=-NCPU)["rgb8"]
    ig = g.render(80, 60, 32, seed=1)
    a, b = ig.reshape(-1, 3).astype(np.float64), io.reshape(-1, 3).astype(np.float64)
    mre = np.abs(a.mean(0) - b.mean(0)) / b.mean(0)
    parity_log("gpu/dielectric/frame", psnr=psnr(ig, io), mre=mre)
    assert psnr(ig, io) >= 38.0 and (mre < 0.015).all()


def test_glass_sphere_transmittance_closed_form(rtb):
    g = rtb.Scene.from_toml_string(AXIS_SCENE)
    n, spp = 400_000, 1 << 19
    si = np.random.default_rng(2).choice(spp, n, replace=False)
    L = g.sample_radiance(AXIS_W, AXIS_W, spp, np.full(n, 1000), np.full(n, 1000), si, seed=3).astype(np.float64)
    assert np.abs(L.mean(0) / AXIS_WANT - 1).max() < 0.01, L.mean(0)


def test_balance_estimator_has_the_same_mean(rtb, scenes, parity_log):
    g, _ = scenes
    W, H, spp, n = 200, 150, 1024, 300_000
    rng = np.random.default_rng(3)
    px, py, si = rng.integers(0, W, n), rng.integers(0, H, n), rng.integers(0, spp, n)
    nee = g.sample_radiance(W, H, spp, px, py, si, seed=1).astype(np.float64)
    bal = g.sample_radiance(W, H, spp, px, py, si, seed=1, estimator=rtb.EST_MIS_BALANCE).astype(np.float64)
    se = np.sqrt(nee.var(0) / n + bal.var(0) / n)
    parity_log("gpu/dielectric/mis_balance", paths=n, mean_nee=nee.mean(0), mean_balance=bal.mean(0), se=se)
    assert (np.abs(nee.mean(0) - bal.mean(0)) < 4 * se).all(), (nee.mean(0), bal.mean(0), se)
    f = g.render(200, 150, 64, seed=5, estimator=rtb.EST_MIS_BALANCE).astype(int)
    assert abs(f.mean() - g.render(200, 150, 64, seed=6).astype(int).mean()) < 0.02 * f.mean()


RAY_KEYS = ("samples", "rays_primary", "rays_extension", "rays_shadow", "rays_bvh", "shadow_bvh")


def test_scheduling_does_not_change_the_frame(rtb, scenes, monkeypatch):
    g, _ = scenes
    W, H, spp = 200, 150, 64
    monkeypatch.setenv("RTB_INLINE_TAIL", "0")
    ref = g.render(W, H, spp, seed=17).astype(int)
    base = g.stats()
    assert base["rays_extension"] > 0
    monkeypatch.delenv("RTB_INLINE_TAIL")
    for kw in ({}, {"pool_paths": 1024}, {"pool_paths": 6000}):   # the default inline tail; two pool sizes
        f = g.render(W, H, spp, seed=17, **kw).astype(int)
        st = g.stats()
        assert np.abs(f - ref).max() <= 1, kw
        assert all(st[k] == base[k] for k in RAY_KEYS), (kw, st, base)   # the same rays, only their schedule differs
    # two emulated ranks, untiled: the union of their tiles is the world = 1 frame
    out = np.zeros((H, W, 3), dtype=np.uint8)
    for r in range(2):
        g.render(W, H, spp, seed=17, rank=r, world=2, out=out)
    assert np.abs(out.astype(int) - ref).max() <= 1


def test_progressive_and_denoised(rtb, scenes):
    g, _ = scenes
    W, H, spp, seed = 200, 150, 64, 8
    ref = g.render(W, H, spp, seed=seed)
    job = rtb.RenderJob(g, W, H, spp, seed=seed, passes=4)
    frames = list(job.frames())
    assert not job.close()
    assert np.abs(frames[-1][1].astype(int) - ref.astype(int)).max() <= 1
    dn = g.render(W, H, spp, seed=seed, denoise=True)
    assert dn.shape == ref.shape and abs(dn.astype(float).mean() - ref.astype(float).mean()) < 0.05 * ref.mean()


def test_guides_look_through_glass(rtb):
    # the pixel looking through the centre of a glass sphere is guided by what it shows: the wall behind, times the tint of
    # both crossings
    text = """
[camera]
pos = [0.0, 0.0, 10.0]
dir = [0.0, 0.0, -1.0]
[[objects]]
brdf = { type = "diffuse", kd = [0.5, 0.6, 0.7] }
geometry = { type = "plane", pos = [0.0, 0.0, -5.0], n = [0.0, 0.0, 1.0] }
[[objects]]
brdf = { type = "dielectric", ior = 1.5, tint = [0.9, 0.8, 0.5] }
geometry = { type = "sphere", pos = [0.0, 0.0, 0.0], r = 2.0 }
[[objects]]
emitted = [4.0, 4.0, 4.0]
brdf = { type = "diffuse", kd = [0.0, 0.0, 0.0] }
geometry = { type = "sphere", pos = [0.0, 8.0, 0.0], r = 1.0 }
"""
    g = rtb.Scene.from_toml_string(text)
    gb = g.gbuffer(65, 65)
    assert gb["obj"][32, 32] == 0
    assert np.allclose(gb["albedo"][32, 32], [0.5 * 0.81, 0.6 * 0.64, 0.7 * 0.25], rtol=1e-5)
    assert gb["depth"][32, 32] == pytest.approx(15.0, rel=1e-3)
