"""Adaptive sampling without a GPU: the rtb_adaptive layout, option validation on a host-only scene, the per-pixel rule of
k_adapt (adaptive_rule.cuh compiled into a host harness) against a numpy restatement, and the server's "noise" field."""
import asyncio
import ctypes as C
import json
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT, scene_path

NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")


def test_adaptive_layout_matches_header(rtb, tmp_path):
    from raytracer_server_b200 import _abi

    src = tmp_path / "layout.c"
    src.write_text("""#include <stdio.h>
#include <stddef.h>
#include "rtb200.h"
int main(void) {
    printf("%zu %zu %zu %zu %zu %zu\\n", sizeof(rtb_adaptive), offsetof(rtb_adaptive, target_levels), offsetof(rtb_adaptive, pass_spp),
           offsetof(rtb_adaptive, min_spp), offsetof(rtb_adaptive, reserved), sizeof(rtb_params));
    return 0;
}
""")
    exe = tmp_path / "layout"
    subprocess.run(["/usr/bin/gcc", "-std=c99", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    v = [int(x) for x in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()]
    A = _abi.Adaptive
    assert v == [C.sizeof(A), A.target_levels.offset, A.pass_spp.offset, A.min_spp.offset, A.reserved.offset, 56]


BAD = [  # (spp, world, target_levels, pass_spp, min_spp, reserved) -> the field the message must name
    ((64, 1, float("nan"), 16, 32, 0), "target_levels"),
    ((64, 1, float("inf"), 16, 32, 0), "target_levels"),
    ((64, 1, -0.5, 16, 32, 0), "target_levels"),
    ((64, 1, 1.0, 0, 32, 0), "pass_spp"),
    ((64, 1, 1.0, -16, 32, 0), "pass_spp"),
    ((64, 1, 1.0, 6, 36, 0), "pass_spp"),
    ((72, 1, 1.0, 16, 32, 0), "spp"),
    ((64, 1, 1.0, 16, 24, 0), "min_spp"),
    ((64, 1, 1.0, 16, 16, 0), "min_spp"),
    ((64, 1, 1.0, 16, 80, 0), "min_spp"),
    ((64, 1, 1.0, 16, 32, 1), "reserved"),
    ((64, 2, 1.0, 16, 32, 0), "world"),
]


def _opts(rtb, target, pass_spp, min_spp, reserved):
    o = rtb.Adaptive()
    o.target_levels, o.pass_spp, o.min_spp, o.reserved = target, pass_spp, min_spp, reserved
    return o


@pytest.mark.parametrize("case", BAD, ids=[f"{f}-{i}" for i, (_, f) in enumerate(BAD)])
def test_invalid_options_are_refused_on_the_host(rtb, case):
    from raytracer_server_b200 import _abi

    (spp, world, target, pass_spp, min_spp, reserved), field = case
    sc = rtb.Scene.from_toml(scene_path("cornell_box"), device=-1)
    p = rtb.make_params(64, 48, spp, world=world)
    o = _opts(rtb, target, pass_spp, min_spp, reserved)
    frame = (C.c_uint8 * (64 * 48 * 3))()
    assert _abi.lib().rtb_render_adaptive(sc._h, C.byref(p), C.byref(o), frame, None, None, None) == _abi.RTB_EINVAL
    assert field in _abi.last_error()
    job = C.c_void_p()
    assert _abi.lib().rtb_job_begin_adaptive(sc._h, C.byref(p), C.byref(o), C.byref(job)) == _abi.RTB_EINVAL
    assert field in _abi.last_error() and not job.value


def test_valid_options_need_a_device(rtb):
    from raytracer_server_b200 import _abi

    sc = rtb.Scene.from_toml(scene_path("cornell_box"), device=-1)
    frame = (C.c_uint8 * (64 * 48 * 3))()
    job = C.c_void_p()
    for spp, target, pass_spp, min_spp in [(64, 1.0, 16, 32), (64, 0.0, 16, 64), (4096, 2.0, 16, 64), (8, 0.5, 4, 8)]:
        p = rtb.make_params(64, 48, spp)
        o = _opts(rtb, target, pass_spp, min_spp, 0)
        assert _abi.lib().rtb_render_adaptive(sc._h, C.byref(p), C.byref(o), frame, None, None, None) == _abi.RTB_ECUDA
        assert _abi.lib().rtb_job_begin_adaptive(sc._h, C.byref(p), C.byref(o), C.byref(job)) == _abi.RTB_ECUDA
    assert rtb.make_adaptive(4096, target_levels=1.0).min_spp == 64 and rtb.make_adaptive(32, target_levels=1.0).min_spp == 32


# ---- the per-pixel rule (adapt_pixel, csrc/adaptive_rule.cuh) ----------------------------------------------------------
HARNESS = r"""
#include <cstdio>
#include "adaptive_rule.cuh"
// stdin: records of 20 floats {sub[4] as float4, inv_n, mean, M2, B}; stdout: 7 floats {sub[s].w, mean, M2, err} per record
int main() {
    float in[20];
    while (fread(in, sizeof(float), 20, stdin) == 20) {
        float4 sub[4];
        for (int s = 0; s < 4; ++s) sub[s] = make_float4(in[4 * s], in[4 * s + 1], in[4 * s + 2], in[4 * s + 3]);
        float2 mom = make_float2(in[17], in[18]);
        const float err = rtb::adapt_pixel(sub, in[16], mom, (int)in[19]);
        const float out[7] = {sub[0].w, sub[1].w, sub[2].w, sub[3].w, mom.x, mom.y, err};
        fwrite(out, sizeof(float), 7, stdout);
    }
    return 0;
}
"""


def restated(sub, inv_n, mean, m2, B):
    """the rule as the header states it, in float64"""
    lum = 0.2126 * sub[..., 0] + 0.7152 * sub[..., 1] + 0.0722 * sub[..., 2]
    m = 0.25 * np.clip((lum - sub[..., 3]) * inv_n[:, None], 0.0, 1.0).sum(1)
    delta = m - mean
    mean = mean + delta / B
    m2 = m2 + delta * (m - mean)
    mu = np.clip(mean, 0.0, 1.0)
    with np.errstate(divide="ignore", invalid="ignore"):
        sigma = np.sqrt(np.maximum(m2, 0.0) / (B - 1) / B)
        err = 255.0 * (np.minimum(mu + sigma, 1.0) ** (1 / 2.2) - mu ** (1 / 2.2))
    return lum, mean, m2, np.where(B < 2, np.inf, err)


@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    d = tmp_path_factory.mktemp("adapt_rule")
    (d / "h.cu").write_text(HARNESS)
    exe = d / "h"
    subprocess.run([NVCC, "-std=c++17", "-O2", "-ccbin", "/usr/bin/g++", "-I", os.path.join(ROOT, "raytracer-server_b200", "csrc"),
                    str(d / "h.cu"), "-o", str(exe)], check=True)

    def run(rec):
        out = subprocess.run([str(exe)], input=np.ascontiguousarray(rec, dtype=np.float32).tobytes(), capture_output=True, check=True).stdout
        return np.frombuffer(out, dtype=np.float32).reshape(-1, 7).astype(np.float64)

    return run


def _cases(rng):
    n = 4000
    pass_spp = rng.choice([4, 16, 64], n)
    B = rng.integers(1, 40, n)
    inv_n = 4.0 / pass_spp
    prev = rng.uniform(0, 3, (n, 4)) * (B[:, None] - 1) * pass_spp[:, None] / 4   # luminance sums after the previous pass
    gain = rng.uniform(-0.1, 1.6, (n, 4, 3)) * (pass_spp[:, None, None] / 4)
    sub = np.empty((n, 4, 4))
    sub[..., :3] = prev[..., None] + gain
    sub[..., 3] = prev
    mean = rng.uniform(-0.05, 1.1, n)
    m2 = rng.uniform(0, 2, n) * (B > 1)
    # edge rows: mu = 0 (black, nothing ever added) | sigma = 0 (same batch value every pass) | mu + sigma > 1 | B = 2
    k = np.arange(n) % 8
    black = k == 0
    sub[black] = 0.0
    mean[black] = 0.0
    m2[black] = 0.0
    flat = k == 1
    sub[flat, :, :3] = (sub[flat, :, 3] + 0.5 / inv_n[flat, None])[..., None]
    mean[flat] = 0.5
    m2[flat] = 0.0
    bright = k == 2
    mean[bright] = 0.98
    m2[bright] = 5.0
    B[k == 3] = 2
    B[k == 4] = 1
    rec = np.concatenate([sub.reshape(n, 16), inv_n[:, None], mean[:, None], m2[:, None], B[:, None]], axis=1).astype(np.float32)
    return rec, k


def test_adapt_pixel_matches_the_stated_rule(harness):
    rng = np.random.default_rng(5)
    rec, k = _cases(rng)
    got = harness(rec)
    r = rec.astype(np.float64)
    sub, inv_n, mean, m2, B = r[:, :16].reshape(-1, 4, 4), r[:, 16], r[:, 17], r[:, 18], r[:, 19]
    lum, mean1, m21, err = restated(sub, inv_n, mean, m2, B)
    np.testing.assert_allclose(got[:, :4], lum, rtol=1e-5, atol=1e-4)
    np.testing.assert_allclose(got[:, 4], mean1, rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(got[:, 5], m21, rtol=1e-4, atol=1e-5)
    one = B < 2
    assert np.isinf(got[one, 6]).all()
    np.testing.assert_allclose(got[~one, 6], err[~one], rtol=1e-3, atol=2e-3)
    # the edges behave as stated
    assert (got[k == 0, 6][B[k == 0] >= 2] == 0).all()                      # mu = 0, sigma = 0: no error
    assert np.abs(got[k == 1, 6][B[k == 1] >= 2]).max() < 1e-2              # same batch value every pass: sigma = 0
    bright = (k == 2) & (B >= 2)
    np.testing.assert_allclose(got[bright, 6], 255.0 * (1.0 - np.clip(mean1[bright], 0, 1) ** (1 / 2.2)), rtol=1e-3, atol=2e-3)
    assert np.isfinite(got[k == 3, 6]).all() and (got[~one, 6] >= 0).all()


def test_welford_over_passes_is_the_sample_statistic(harness):
    # B passes fed one after the other: (mean, M2) equal numpy's mean and sum of squared deviations of the batch values
    rng = np.random.default_rng(9)
    pass_spp, B = 16, 12
    batch = rng.uniform(0, 1, (B, 4))                 # per sub-pixel luminance means of each pass
    prev = np.zeros(4)
    mean, m2 = 0.0, 0.0
    for b in range(B):
        sums = prev + batch[b] * pass_spp / 4
        sub = np.zeros((4, 4))
        sub[:, :3] = sums[:, None]                      # grey: luminance = the channel value
        sub[:, 3] = prev
        rec = np.concatenate([sub.reshape(16), [4.0 / pass_spp, mean, m2, b + 1]])[None]
        out = harness(rec)[0]
        prev, mean, m2, err = out[:4], out[4], out[5], out[6]
    m = batch.mean(1)
    assert mean == pytest.approx(m.mean(), rel=1e-5)
    assert m2 == pytest.approx(((m - m.mean()) ** 2).sum(), rel=1e-4)
    mu, sigma = m.mean(), m.std(ddof=1) / np.sqrt(B)
    assert err == pytest.approx(255.0 * ((mu + sigma) ** (1 / 2.2) - mu ** (1 / 2.2)), rel=1e-3)


# ---- server: "noise" selects an adaptive job -----------------------------------------------------------------------
websockets = pytest.importorskip("websockets")


class _Job:
    def __init__(self):
        self.closed = False

    def messages(self):
        yield bytes([0, 1, 0, 0, 0, 0, 1, 2, 3])

    def stop(self):
        pass

    def close(self):
        self.closed = True
        return False


def _serve(factory):
    from test_server_protocol import run_server

    from raytracer_server_b200.server import Server

    return run_server(Server({}, width=1, height=1, job_factory=factory, log=lambda *a: None))


def _send(port, req, expect_close=False):
    async def go():
        async with websockets.connect(f"ws://127.0.0.1:{port}") as ws:
            await ws.send(json.dumps(req))
            if expect_close:
                with pytest.raises(websockets.ConnectionClosed):
                    await asyncio.wait_for(ws.recv(), timeout=5)
                return ws.close_code
            return await asyncio.wait_for(ws.recv(), timeout=5)

    return asyncio.run(go())


def test_noise_request_reaches_the_factory_as_adaptive_options(rtb):
    calls = []

    def factory(scene, spp, passes=1, **kw):
        calls.append((scene, spp, passes, kw))
        return _Job()

    port, stop = _serve(factory)
    try:
        for spp, noise in [(4100, 1.5), (100, 2), (40, 0), (20, 1.0), (-5, 1.0)]:
            assert _send(port, {"type": "render", "scene": "cornell_box", "spp": spp, "noise": noise}) == bytes([0, 1, 0, 0, 0, 0, 1, 2, 3])
    finally:
        stop()
    assert calls[0] == ("cornell_box", 4096, 1, {"adaptive": {"target_levels": 1.5, "pass_spp": 16, "min_spp": 64}})
    assert calls[1] == ("cornell_box", 96, 1, {"adaptive": {"target_levels": 2.0, "pass_spp": 16, "min_spp": 64}})
    assert calls[2] == ("cornell_box", 32, 1, {"adaptive": {"target_levels": 0.0, "pass_spp": 16, "min_spp": 32}})
    # a budget below two passes: a plain job, called the old way
    assert calls[3] == ("cornell_box", 20, 1, {}) and calls[4] == ("cornell_box", -5, 1, {})


def test_request_without_noise_keeps_the_old_factory_signature(rtb):
    calls = []

    def factory(scene, spp, passes=1):
        calls.append((scene, spp, passes))
        return _Job()

    port, stop = _serve(factory)
    try:
        _send(port, {"type": "render", "scene": "cornell_box", "spp": 64, "passes": 3})
    finally:
        stop()
    assert calls == [("cornell_box", 64, 3)]


@pytest.mark.parametrize("noise", ["1", True, None, -1, -0.5, [1], 1e400])
def test_bad_noise_closes_the_connection(rtb, noise):
    calls = []
    port, stop = _serve(lambda *a, **kw: calls.append(a) or _Job())
    try:
        assert _send(port, {"type": "render", "scene": "cornell_box", "spp": 64, "noise": noise}, expect_close=True) == 1007
    finally:
        stop()
    assert calls == []
