"""The denoiser on the GPU: guides (rtb_scene_gbuffer), the filter alone (rtb_denoise_image) against its numpy twin,
denoised whole frames, jobs and the server's "denoise" request, and the quality it buys against the 4096-spp goldens.

Frames of two runs differ by the order of the fp32 atomics; comparisons between runs allow one level per pixel."""
import asyncio
import json
import os

import numpy as np
import pytest

from conftest import ROOT
from parity_metrics import compare_regions, psnr
from test_denoise_cpu import restated_filter

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(ROOT, "tests", "golden", "converged")


def specular_objects(g):
    return {i for i in range(g.info.n_objects) if g.object(i)["brdf"] == 1}


@pytest.mark.parametrize("name", ["cornell_box", "cubes", "flying_unicorn"])
@pytest.mark.parametrize("accel", [0, 1])
def test_guides_follow_the_primary_rays(gpu_scene, oracle_scene, parity_log, name, accel):
    g = gpu_scene(name)
    W, H = 200, 150
    gb = g.gbuffer(W, H, accel=accel)
    hits = [g.trace_primary(W, H, s & 1, s >> 1) for s in range(4)]
    obj = np.stack([h["obj"] for h in hits]).reshape(4, H, W)
    t = np.stack([h["t"] for h in hits]).reshape(4, H, W).astype(np.float64)
    spec = specular_objects(g)
    agree = (obj == obj[0]).all(0) & (obj[0] >= 0) & ~np.isin(obj[0], list(spec))
    meshes = {i for i in range(g.info.n_objects) if g.object(i)["geometry"] == 2}
    # the reference's octrees need not return the nearest triangle: in that mode only analytic hits are bound to be the same
    exact = agree & (~np.isin(obj[0], list(meshes)) if accel == 1 else True)
    assert exact.sum() > 0.5 * W * H
    same_obj = gb["obj"][exact] == obj[0][exact]
    rel = np.abs(gb["depth"][exact] - t.mean(0)[exact]) / t.mean(0)[exact]
    n = gb["normal"]
    length = np.linalg.norm(n, axis=2)
    dirs = g_dirs(oracle_scene(name), W, H)
    facing = (n * dirs).sum(2)
    parity_log(f"gpu/denoise/guides/{name}-accel{accel}", agreeing_pixels=int(agree.sum()), checked=int(exact.sum()),
               obj_match=float(same_obj.mean()), depth_rel_max=float(rel.max()), normal_len_err_max=float(np.abs(length[agree] - 1).max()),
               facing_max=float(facing[agree].max()))
    assert same_obj.all()
    assert rel.max() <= 1e-5
    assert np.abs(length[agree] - 1).max() < 1e-5 and (facing[agree] < 0).all()
    if accel == 1:
        assert (gb["obj"][agree] == obj[0][agree]).mean() > 0.99
    for s in spec:   # mirror pixels report the object seen in the mirror
        m = (obj == s).all(0)
        if m.any():
            seen = gb["obj"][m]
            parity_log(f"gpu/denoise/guides/{name}-accel{accel}/mirror{s}", pixels=int(m.sum()), frac_other=float((seen != s).mean()),
                       frac_hit=float((seen >= 0).mean()))
            hit = seen >= 0
            assert (seen != s).mean() > 0.99 and (gb["depth"][m][hit] > t.mean(0)[m][hit]).all()


def g_dirs(o, W, H):
    _, dirs = o.primary_rays(W, H, 0, 0, 0.0, 0.0)
    return np.asarray(dirs, dtype=np.float64).reshape(H, W, 3)


def linear_frame(g, W, H, seeds, spp):
    """mean of len(seeds) frames decoded to linear rgb, and the luminance variance of that mean"""
    fr = np.stack([(g.render(W, H, spp, seed=s).astype(np.float64) / 255.0) ** 2.2 for s in seeds])
    lum = 0.2126 * fr[..., 0] + 0.7152 * fr[..., 1] + 0.0722 * fr[..., 2]
    return fr.mean(0).astype(np.float32), (lum.var(0, ddof=1) / len(seeds)).astype(np.float32)


def test_filter_matches_its_numpy_twin(gpu_scene, rtb, parity_log):
    g = gpu_scene("flying_unicorn")
    W, H = 160, 120
    color, variance = linear_frame(g, W, H, (1, 2, 3, 4), 16)   # 64 spp in all
    gb = g.gbuffer(W, H)
    inputs = dict(color=color, variance=variance, albedo=gb["albedo"], normal=gb["normal"], depth=gb["depth"], obj=gb["obj"])
    got = rtb.denoise_image(**inputs)
    again = rtb.denoise_image(**inputs)
    want = restated_filter(inputs, 5)
    d = np.abs(got - want)
    parity_log("gpu/denoise/twin", max_abs=float(d.max()), mean_change=float(np.abs(got - color).mean()))
    assert got.tobytes() == again.tobytes()
    assert d.max() <= 1e-4
    assert np.abs(got - color).mean() > 1e-3


@pytest.mark.parametrize("name,accel", [("cornell_box", 0), ("flying_unicorn", 0), ("flying_unicorn", 1)])
def test_levels_zero_is_the_plain_resolve(gpu_scene, rtb, parity_log, name, accel):
    g = gpu_scene(name)
    W, H, spp, seed = 200, 150, 64, 5
    raw = g.render(W, H, spp, seed=seed, accel=accel)
    dn = g.render(W, H, spp, seed=seed, accel=accel, denoise=rtb.make_denoise(0))
    d = np.abs(raw.astype(int) - dn.astype(int))
    parity_log(f"gpu/denoise/levels0/{name}-accel{accel}", max_level_diff=int(d.max()), frac_diff=float((d > 0).mean()))
    assert d.max() <= 1


# Margins set before any measurement: +6 dB at 16 spp (4x the samples), at most -0.3 dB at 1024 spp, 50x50-tile mean error at
# most 0.5 % worse than the raw frame's.  Measured on a B200 (profiles/denoise_b200.json): +7.4 to +9.4 dB at 16 spp, +4.4 to
# +5.1 dB at 1024 spp, tile error +0.04 % at 16 spp and +0.04 to +0.08 % at 1024 spp.  Every value goes to the parity log.
@pytest.mark.parametrize("name", ["cornell_box", "cubes", "flying_unicorn"])
def test_quality_against_the_golden(gpu_scene, parity_log, name):
    g = gpu_scene(name)
    gold = np.load(os.path.join(GOLDEN, f"{name}_nee_600x450_4096spp_seed7.npz"))["rgb8"]
    W, H, seed = 600, 450, 13
    res = {}
    for spp in (16, 1024):
        raw = g.render(W, H, spp, seed=seed)
        dn = g.render(W, H, spp, seed=seed, denoise=True)
        res[spp] = dict(psnr_raw=psnr(raw, gold), psnr_denoised=psnr(dn, gold), region_raw=float(compare_regions(raw, gold)[0]),
                        region_denoised=float(compare_regions(dn, gold)[0]))
        parity_log(f"gpu/denoise/quality/{name}/{spp}spp", **res[spp])
    assert res[16]["psnr_denoised"] >= res[16]["psnr_raw"] + 6.0
    assert res[1024]["psnr_denoised"] >= res[1024]["psnr_raw"] - 0.3
    for spp in (16, 1024):
        assert res[spp]["region_denoised"] <= res[spp]["region_raw"] + 0.005


def test_denoised_jobs(gpu_scene, rtb, parity_log):
    g = gpu_scene("cornell_box")
    W, H, spp, seed = 200, 150, 64, 8
    ref = g.render(W, H, spp, seed=seed, denoise=True)
    job = rtb.RenderJob(g, W, H, spp, seed=seed, passes=4, denoise=True)
    frames = list(job.frames())
    assert not job.close()
    assert [i for i, _ in frames] == [0, 1, 2, 3]
    d_prog = np.abs(frames[-1][1].astype(int) - ref.astype(int))
    # a single pass: one band, sent as the reference's records
    job = rtb.RenderJob(g, W, H, spp, seed=seed, denoise=True)
    frame = np.zeros((H, W, 3), dtype=np.uint8)
    for m in job.messages():
        n, x, y = m[1], int.from_bytes(m[2:4], "little"), int.from_bytes(m[4:6], "little")
        frame[y, x: x + n] = np.frombuffer(m[6:], dtype=np.uint8).reshape(n, 3)
    assert not job.close()
    d_one = np.abs(frame.astype(int) - ref.astype(int))
    parity_log("gpu/denoise/job", progressive_max_level_diff=int(d_prog.max()), single_max_level_diff=int(d_one.max()))
    assert d_prog.max() <= 1 and d_one.max() <= 1


def test_denoised_adaptive_job(gpu_scene, rtb, parity_log):
    g = gpu_scene("cornell_box")
    gold = np.load(os.path.join(GOLDEN, "cornell_box_nee_600x450_4096spp_seed7.npz"))["rgb8"]
    W, H, spp, seed = 600, 450, 1024, 13
    opts = dict(target_levels=4.0, pass_spp=16, min_spp=32)
    job = rtb.RenderJob(g, W, H, spp, seed=seed, adaptive=opts, denoise=True)
    frames = list(job.frames())
    assert not job.close()
    raw, _, _ = g.render_adaptive(W, H, spp, seed=seed, **opts)
    pd, pr = psnr(frames[-1][1], gold), psnr(raw, gold)
    parity_log("gpu/denoise/adaptive_job", passes=len(frames), psnr_denoised=pd, psnr_raw=pr)
    assert pd >= pr


def test_server_denoise_request(gpu_scene, rtb):
    websockets = pytest.importorskip("websockets")
    from test_server_protocol import run_server

    from raytracer_server_b200.server import Server

    g = gpu_scene("cornell_box")
    W, H, seed = 120, 90, 17
    calls = []

    def factory(scene, spp, passes=1, denoise=False):
        calls.append((spp, passes, denoise))
        return rtb.RenderJob(g, W, H, spp, passes=passes, seed=seed, denoise=denoise or None)

    port, stop = run_server(Server({}, width=W, height=H, job_factory=factory, log=lambda *a: None))

    async def go():
        frame = np.zeros((H, W, 3), dtype=np.uint8)
        seen = 0
        async with websockets.connect(f"ws://127.0.0.1:{port}", max_size=1 << 20) as ws:
            await ws.send(json.dumps({"type": "render", "scene": "cornell_box", "spp": 64, "denoise": True}))
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
    assert calls == [(64, 1, True)]
    ref = g.render(W, H, 64, seed=seed, denoise=True)
    assert np.abs(frame.astype(int) - ref.astype(int)).max() <= 1


def test_world_above_one_is_refused(gpu_scene, rtb):
    g = gpu_scene("cornell_box")
    with pytest.raises(rtb.RtbError) as e:
        g.render(64, 48, 16, world=2, denoise=True)
    assert e.value.code == rtb.RTB_EINVAL and "world" in str(e.value)
