"""Next-event estimation over every emitter (EST_NEE_ALL_LIGHTS, k_shade MODE 4 / 5) on the GPU: per-path radiance against
the f64 oracle under shared random numbers, the single-sphere-light identity with EST_NEE, unbiasedness against the sum of
one-light renders, and the estimator through every render path."""
import asyncio
import json
import os

import numpy as np
import pytest

from conftest import SCENES, scene_path
from parity_metrics import path_error
from test_gpu_dielectric import GLASS_SCENE

pytestmark = pytest.mark.gpu
ASSETS = os.path.join(SCENES, "assets")
CORNELL = open(scene_path("cornell_box")).read()
LIGHT_B = """
[[objects]]
emitted = [6.0, 12.0, 30.0]
brdf = { type = "diffuse", kd = [0.0, 0.0, 0.0] }
geometry = { type = "sphere", pos = [20.0, 60.0, 60.0], r = 6.0 }
"""
CUBE_LIGHT = """
[[objects]]
emitted = [8.0, 5.0, 2.0]
brdf = { type = "diffuse", kd = [0.0, 0.0, 0.0] }
geometry = { type = "cube", pos = [70.0, 55.0, 50.0], size = 6.0 }
transforms = [ { rotate_y = 0.6 }, { rotate_x = 0.4 }, { scale = 1.5 } ]
"""
# behind the camera: only bounce rays meet it
PLANE_LIGHT = """
[[objects]]
emitted = [0.4, 0.3, 0.2]
brdf = { type = "diffuse", kd = [0.0, 0.0, 0.0] }
geometry = { type = "plane", pos = [0.0, 0.0, 300.0], n = [0.0, 0.0, -1.0] }
"""
SCENES_3 = {
    "two_spheres": CORNELL + LIGHT_B,
    "sphere_and_mesh": CORNELL + CUBE_LIGHT,
    "plane": CORNELL + LIGHT_B + PLANE_LIGHT,
    "glass": GLASS_SCENE + LIGHT_B,
}


@pytest.fixture(scope="module")
def oracle3(oracle_mod):
    """the f64 glass oracle with estimator 3 (tests/lights_oracle.py); oracle_mod builds the oracle whose entry points it shares"""
    import lights_oracle

    lights_oracle.lib()
    return lights_oracle


@pytest.fixture(scope="module")
def scenes(rtb):
    cache = {}

    def get(name):
        if name not in cache:
            cache[name] = rtb.Scene.from_toml_string(SCENES_3[name], assets_dir=ASSETS)
        return cache[name]

    return get


@pytest.mark.parametrize("name, octree", [("two_spheres", False), ("sphere_and_mesh", False), ("sphere_and_mesh", True),
                                          ("plane", False), ("glass", False)])
def test_path_radiance_matches_the_oracle(rtb, oracle3, scenes, parity_log, name, octree):
    g = scenes(name)
    o = oracle3.OracleScene.from_toml_string(SCENES_3[name], ASSETS)
    assert len(g.lights()["objects"]) == 2
    W, H, spp, n = 200, 150, 32, 20000
    rng = np.random.default_rng(31)
    px, py, si = rng.integers(0, W, n), rng.integers(0, H, n), rng.integers(0, spp, n)
    o.set_modes(oracle3.ACCEL_OCTREE_FAITHFUL if octree else oracle3.ACCEL_EXACT, 3)
    Lo = o.sample_radiance(W, H, spp, 9, px, py, si)
    Lg = g.sample_radiance(W, H, spp, px, py, si, seed=9, estimator=rtb.EST_NEE_ALL_LIGHTS,
                           accel=rtb.ACCEL_OCTREE_REFERENCE if octree else 0).astype(np.float64)
    fin = np.isfinite(Lo).all(axis=1) & np.isfinite(Lg).all(axis=1)
    err = path_error(Lg[fin], Lo[fin])
    parity_log(f"gpu/lights/path_radiance/{name}{'_octree' if octree else ''}", paths=n, err_median=np.median(err),
               frac_beyond_1e3=(err > 1e-3).mean(), mean_gpu=Lg[fin].mean(0), mean_oracle=Lo[fin].mean(0))
    assert fin.mean() > 0.99 and Lo[fin].sum() > 0
    assert np.median(err) < 2e-5 and (err > 1e-3).mean() < 0.03


@pytest.mark.parametrize("name", ["cornell_box", "cubes", "flying_unicorn"])
def test_single_sphere_light_equals_nee(rtb, gpu_scene, parity_log, name):
    g = gpu_scene(name)
    W, H, spp, n = 600, 450, 64, 100000
    rng = np.random.default_rng(5)
    px, py, si = rng.integers(0, W, n), rng.integers(0, H, n), rng.integers(0, spp, n)
    nee = g.sample_radiance(W, H, spp, px, py, si, seed=4).astype(np.float64)
    alll = g.sample_radiance(W, H, spp, px, py, si, seed=4, estimator=rtb.EST_NEE_ALL_LIGHTS).astype(np.float64)
    d = np.abs(alll - nee).max(axis=1)
    parity_log(f"gpu/lights/single_light/{name}", paths=n, median=np.median(d), frac_within_1e4=(d <= 1e-4).mean())
    assert np.median(d) < 1e-6 and (d <= 1e-4).mean() >= 0.999


def _sub_means(rtb, g, W, H, spp, seed, estimator):
    """linear sub-pixel means [H, W, 4, 3] of a render_device call"""
    import torch

    from raytracer_server_b200 import sharding

    n = sharding.local_pixels(W, H, 0, 1)
    rgb = torch.zeros(n * 3, dtype=torch.uint8, device="cuda:0")
    sub = torch.zeros(n * 4 * 4, dtype=torch.float32, device="cuda:0")
    g.render_device(rtb.make_params(W, H, spp, seed=seed, estimator=estimator), rgb.data_ptr(), sub.data_ptr())
    s = sub.cpu().numpy().reshape(n, 4, 4)[:, :, :3].astype(np.float64) / (spp // 4)
    xy = sharding.tile_map(W, H, 0, 1)
    ok = xy[:, 0] >= 0
    out = np.zeros((H, W, 4, 3))
    out[xy[ok, 1], xy[ok, 0]] = s[ok]
    return out


def _blocks(img):
    H, W = img.shape[:2]
    return img[: H // 8 * 8, : W // 8 * 8].reshape(H // 8, 8, W // 8, 8, -1).mean(axis=(1, 3))


def test_unbiased_against_one_light_renders(rtb, parity_log):
    # the light estimator 0 sees with only A emitting plus the light it sees with only B emitting is what estimator 3 sees
    # with both: compared per 8x8 block against the spread between two seeds of the same estimator-3 render
    both = CORNELL + LIGHT_B
    only_a = CORNELL + LIGHT_B.replace("emitted = [6.0, 12.0, 30.0]", "emitted = [0.0, 0.0, 0.0]")
    only_b = CORNELL.replace("emitted = [50.0, 50.0, 50.0]", "emitted = [0.0, 0.0, 0.0]") + LIGHT_B
    W, H, spp = 160, 120, 1024
    g = rtb.Scene.from_toml_string(both)
    e3 = [_blocks(_sub_means(rtb, g, W, H, spp, seed, rtb.EST_NEE_ALL_LIGHTS)) for seed in (1, 2)]
    ga, gb = rtb.Scene.from_toml_string(only_a), rtb.Scene.from_toml_string(only_b)
    assert list(ga.lights()["objects"]) == [8] and list(gb.lights()["objects"]) == [9]
    e0 = _blocks(_sub_means(rtb, ga, W, H, spp, 3, rtb.EST_NEE)) + _blocks(_sub_means(rtb, gb, W, H, spp, 4, rtb.EST_NEE))
    floor = np.abs(e3[0] - e3[1]).mean()
    diff = np.abs((e3[0] + e3[1]) / 2 - e0).mean()
    parity_log("gpu/lights/unbiased", floor=floor, diff=diff, mean_e3=e3[0].mean(), mean_sum=e0.mean())
    assert diff < 2 * floor, (diff, floor)
    assert abs(e3[0].mean() / e0.mean() - 1) < 0.01


def test_every_render_path(rtb, scenes, monkeypatch):
    g = scenes("sphere_and_mesh")
    W, H, spp, seed = 200, 150, 64, 8
    est = rtb.EST_NEE_ALL_LIGHTS
    ref = g.render(W, H, spp, seed=seed, estimator=est).astype(int)
    assert abs(ref.mean() - g.render(W, H, spp, seed=seed).astype(int).mean()) > 1     # the cube adds light
    # progressive job, streamed records
    job = rtb.RenderJob(g, W, H, spp, seed=seed, passes=4, estimator=est)
    frames = list(job.frames())
    assert not job.close() and len(frames) == 4
    assert np.abs(frames[-1][1].astype(int) - ref).max() <= 1
    # adaptive job that never stops early: the uniform frame
    job = rtb.RenderJob(g, W, H, spp, seed=seed, adaptive={"target_levels": 0.0, "pass_spp": 16}, estimator=est)
    frames = list(job.frames())
    assert not job.close()
    assert np.abs(frames[-1][1].astype(int) - ref).max() <= 1
    # denoised render, levels 0 = the resolve through the denoise path
    f0 = g.render(W, H, spp, seed=seed, estimator=est, denoise={"levels": 0})
    assert np.abs(f0.astype(int) - ref).max() <= 1
    dn = g.render(W, H, spp, seed=seed, estimator=est, denoise=True)
    assert abs(dn.astype(float).mean() - ref.mean()) < 0.05 * ref.mean()
    # emulated ranks: the union of world = 2's tiles is the world = 1 frame
    out = np.zeros((H, W, 3), dtype=np.uint8)
    for r in range(2):
        g.render(W, H, spp, seed=seed, rank=r, world=2, out=out, estimator=est)
    assert np.abs(out.astype(int) - ref).max() <= 1
    # the inline tail off: the same frame
    monkeypatch.setenv("RTB_INLINE_TAIL", "0")
    assert np.abs(g.render(W, H, spp, seed=seed, estimator=est).astype(int) - ref).max() <= 1
    monkeypatch.delenv("RTB_INLINE_TAIL")
    # rtb_sample_pixels: the frame's bytes up to the order of the fp32 sums
    from raytracer_server_b200.host import sample_pixels

    rng = np.random.default_rng(2)
    xs, ys = rng.integers(0, W, 300), rng.integers(0, H, 300)
    v = sample_pixels(xs, ys, W, H, spp, g, seed=seed, estimator=est)
    assert np.abs(np.trunc(v).astype(int) - ref[ys, xs]).max() <= 1


def test_glass_scene_frame(rtb, scenes):
    g = scenes("glass")
    W, H, spp = 200, 150, 64
    f = g.render(W, H, spp, seed=5, estimator=rtb.EST_NEE_ALL_LIGHTS).astype(int)
    assert np.abs(g.render(W, H, spp, seed=5, estimator=rtb.EST_NEE_ALL_LIGHTS, pool_paths=6000).astype(int) - f).max() <= 1


def test_server_all_lights_request(rtb, monkeypatch):
    websockets = pytest.importorskip("websockets")
    from test_server_protocol import run_server

    from raytracer_server_b200 import server as S

    g = rtb.Scene.from_toml_string(CORNELL + CUBE_LIGHT)
    W, H, seed = 120, 90, 17
    monkeypatch.setattr(S.random, "getrandbits", lambda k: seed)
    port, stop = run_server(S.Server({"cornell_box": g}, width=W, height=H, log=lambda *a: None))

    async def go():
        frame = np.zeros((H, W, 3), dtype=np.uint8)
        seen = 0
        async with websockets.connect(f"ws://127.0.0.1:{port}", max_size=1 << 20) as ws:
            await ws.send(json.dumps({"type": "render", "scene": "cornell_box", "spp": 64, "all_lights": True}))
            while seen < W * H:
                m = await asyncio.wait_for(ws.recv(), timeout=10.0)
                n, x, y = m[1], int.from_bytes(m[2:4], "little"), int.from_bytes(m[4:6], "little")
                frame[y, x: x + n] = np.frombuffer(m[6:], dtype=np.uint8).reshape(n, 3)
                seen += n
        return frame

    try:
        frame = asyncio.run(go())
    finally:
        stop()
    ref = g.render(W, H, 64, seed=seed, estimator=rtb.EST_NEE_ALL_LIGHTS).astype(int)
    assert np.abs(frame.astype(int) - ref).max() <= 1
    assert (frame.astype(int) == ref).mean() > 0.99
    assert np.abs(g.render(W, H, 64, seed=seed).astype(int) - ref).max() > 1    # the request did not run estimator 0
