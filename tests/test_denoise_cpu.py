"""The denoiser without a GPU: the rtb_denoise layout, option validation on a host-only scene, the filter rule
(denoise_rule.cuh compiled into a host harness) against a numpy restatement and its invariants, and the server's "denoise"
field.  `restated_filter` is also the twin the GPU tests compare rtb_denoise_image with."""
import asyncio
import ctypes as C
import json
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT, scene_path

NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
F = np.float32


def test_denoise_layout_matches_header(rtb, tmp_path):
    from raytracer_server_b200 import _abi

    src = tmp_path / "layout.c"
    src.write_text("""#include <stdio.h>
#include <stddef.h>
#include "rtb200.h"
int main(void) {
    printf("%zu %zu %zu %zu %zu %zu %zu %d\\n", sizeof(rtb_denoise), offsetof(rtb_denoise, levels), offsetof(rtb_denoise, sigma_color),
           offsetof(rtb_denoise, sigma_normal), offsetof(rtb_denoise, sigma_depth), offsetof(rtb_denoise, reserved), sizeof(rtb_params),
           RTB_ABI_VERSION);
    return 0;
}
""")
    exe = tmp_path / "layout"
    subprocess.run(["/usr/bin/gcc", "-std=c99", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    v = [int(x) for x in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()]
    D = _abi.Denoise
    assert v == [C.sizeof(D), D.levels.offset, D.sigma_color.offset, D.sigma_normal.offset, D.sigma_depth.offset, D.reserved.offset, 56, 2]
    d = rtb.make_denoise()
    assert (d.levels, d.sigma_color, d.sigma_normal, d.sigma_depth, list(d.reserved)) == (5, 4.0, 128.0, 1.0, [0, 0, 0, 0])


BAD = [  # (levels, sigma_color, sigma_normal, sigma_depth, reserved, world) -> the field the message must name
    ((-1, 4.0, 128.0, 1.0, (0, 0, 0, 0), 1), "levels"),
    ((9, 4.0, 128.0, 1.0, (0, 0, 0, 0), 1), "levels"),
    ((5, float("nan"), 128.0, 1.0, (0, 0, 0, 0), 1), "sigma_color"),
    ((5, float("inf"), 128.0, 1.0, (0, 0, 0, 0), 1), "sigma_color"),
    ((5, -1.0, 128.0, 1.0, (0, 0, 0, 0), 1), "sigma_color"),
    ((5, 4.0, float("nan"), 1.0, (0, 0, 0, 0), 1), "sigma_normal"),
    ((5, 4.0, -128.0, 1.0, (0, 0, 0, 0), 1), "sigma_normal"),
    ((5, 4.0, 128.0, float("-inf"), (0, 0, 0, 0), 1), "sigma_depth"),
    ((5, 4.0, 128.0, -0.5, (0, 0, 0, 0), 1), "sigma_depth"),
    ((5, 4.0, 128.0, 1.0, (0, 0, 1, 0), 1), "reserved"),
    ((5, 4.0, 128.0, 1.0, (0, 0, 0, 0), 2), "world"),
]


def _denoise(rtb, levels, sc, sn, sz, reserved):
    d = rtb.make_denoise(levels, sigma_color=sc, sigma_normal=sn, sigma_depth=sz)
    d.reserved[:] = list(reserved)
    return d


@pytest.mark.parametrize("case", BAD, ids=[f"{f}-{i}" for i, (_, f) in enumerate(BAD)])
def test_invalid_options_are_refused_on_the_host(rtb, case):
    from raytracer_server_b200 import _abi

    (levels, sc, sn, sz, reserved, world), field = case
    L = _abi.lib()
    sc_ = rtb.Scene.from_toml(scene_path("cornell_box"), device=-1)
    p = rtb.make_params(64, 48, 64, world=world)
    d = _denoise(rtb, levels, sc, sn, sz, reserved)
    frame = (C.c_uint8 * (64 * 48 * 3))()
    for adaptive in (None, rtb.make_adaptive(64, target_levels=1.0)):
        a = C.byref(adaptive) if adaptive is not None else None
        assert L.rtb_render_denoised(sc_._h, C.byref(p), a, C.byref(d), frame, None, None, None) == _abi.RTB_EINVAL
        assert field in _abi.last_error()
        job = C.c_void_p()
        assert L.rtb_job_begin_denoised(sc_._h, C.byref(p), 4, a, C.byref(d), C.byref(job)) == _abi.RTB_EINVAL
        assert field in _abi.last_error() and not job.value
    if field != "world":   # the filter alone checks the same options before it touches a device
        buf = np.zeros(64 * 48 * 3, dtype=np.float32)
        fp = C.POINTER(C.c_float)
        obj = np.zeros(64 * 48, dtype=np.int32)
        assert L.rtb_denoise_image(0, 64, 48, C.byref(d), *[buf.ctypes.data_as(fp)] * 5, obj.ctypes.data_as(C.POINTER(C.c_int32)),
                                   buf.ctypes.data_as(fp)) == _abi.RTB_EINVAL
        assert field in _abi.last_error()


def test_valid_options_need_a_device(rtb):
    from raytracer_server_b200 import _abi

    L = _abi.lib()
    sc = rtb.Scene.from_toml(scene_path("cornell_box"), device=-1)
    frame = (C.c_uint8 * (64 * 48 * 3))()
    job = C.c_void_p()
    p = rtb.make_params(64, 48, 64)
    for levels, sc_, sn, sz in [(0, 0.0, 0.0, 0.0), (5, 4.0, 128.0, 1.0), (8, 1e6, 1.0, 3.0)]:
        d = _denoise(rtb, levels, sc_, sn, sz, (0, 0, 0, 0))
        assert L.rtb_render_denoised(sc._h, C.byref(p), None, C.byref(d), frame, None, None, None) == _abi.RTB_ECUDA
        assert L.rtb_job_begin_denoised(sc._h, C.byref(p), 4, None, C.byref(d), C.byref(job)) == _abi.RTB_ECUDA
    assert L.rtb_scene_gbuffer(sc._h, 64, 48, 0, None, None, None, None) == _abi.RTB_ECUDA


# ---- the filter rule (csrc/denoise_rule.cuh) --------------------------------------------------------------------------
HARNESS = r"""
#include <cstdio>
#include <vector>
#include "denoise_rule.cuh"
using namespace rtb;
// stdin: int32 {W, H, levels}, float32 {sigma_color, sigma_normal, sigma_depth}, then float32 colour[H*W*3], variance[H*W],
// albedo[H*W*3], normal[H*W*3], depth[H*W], int32 obj[H*W]; stdout: float32 out[H*W*3] — rtb_denoise_image on the host
int main() {
    int hdr[3];
    float sig[3];
    if (fread(hdr, 4, 3, stdin) != 3 || fread(sig, 4, 3, stdin) != 3) return 1;
    const int W = hdr[0], H = hdr[1], levels = hdr[2], n = W * H;
    std::vector<float> col(3 * n), var(n), alb(3 * n), nrm(3 * n), dep(n);
    std::vector<int> obj(n);
    if (fread(col.data(), 4, 3 * n, stdin) != (size_t)(3 * n) || fread(var.data(), 4, n, stdin) != (size_t)n ||
        fread(alb.data(), 4, 3 * n, stdin) != (size_t)(3 * n) || fread(nrm.data(), 4, 3 * n, stdin) != (size_t)(3 * n) ||
        fread(dep.data(), 4, n, stdin) != (size_t)n || fread(obj.data(), 4, n, stdin) != (size_t)n) return 1;
    std::vector<float4> ga(n), gn(n), buf0(n), buf1(n);
    for (int i = 0; i < n; ++i) {
        float o;
        memcpy(&o, &obj[i], 4);
        ga[i] = make_float4(alb[3 * i], alb[3 * i + 1], alb[3 * i + 2], dep[i]);
        gn[i] = make_float4(nrm[3 * i], nrm[3 * i + 1], nrm[3 * i + 2], o);
        buf0[i] = demodulate(make_float3(col[3 * i], col[3 * i + 1], col[3 * i + 2]), var[i], make_float3(alb[3 * i], alb[3 * i + 1], alb[3 * i + 2]));
    }
    const DenoiseSigmas s{sig[0], sig[1], sig[2]};
    std::vector<float4>*in = &buf0, *out = &buf1;
    for (int l = 0; l < levels; ++l) {
        for (int y = 0; y < H; ++y)
            for (int x = 0; x < W; ++x) (*out)[y * W + x] = atrous_pixel(in->data(), ga.data(), gn.data(), W, H, x, y, 1 << l, s);
        std::swap(in, out);
    }
    for (int i = 0; i < n; ++i) {
        const float3 v = remodulate((*in)[i], make_float3(alb[3 * i], alb[3 * i + 1], alb[3 * i + 2]));
        const float o3[3] = {v.x, v.y, v.z};
        fwrite(o3, 4, 3, stdout);
    }
    return 0;
}
"""


@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    d = tmp_path_factory.mktemp("denoise_rule")
    (d / "h.cu").write_text(HARNESS)
    exe = d / "h"
    subprocess.run([NVCC, "-std=c++17", "-O2", "-ccbin", "/usr/bin/g++", "-I", os.path.join(ROOT, "raytracer-server_b200", "csrc"),
                    str(d / "h.cu"), "-o", str(exe)], check=True)

    def run(g, levels, sigmas=(4.0, 128.0, 1.0)):
        h, w = g["color"].shape[:2]
        blob = (np.array([w, h, levels], np.int32).tobytes() + np.array(sigmas, F).tobytes() +
                b"".join(np.ascontiguousarray(g[k], F).tobytes() for k in ("color", "variance", "albedo", "normal", "depth")) +
                np.ascontiguousarray(g["obj"], np.int32).tobytes())
        out = subprocess.run([str(exe)], input=blob, capture_output=True, check=True).stdout
        return np.frombuffer(out, dtype=F).reshape(h, w, 3)

    return run


def _lum(c):
    return F(0.2126) * c[..., 0] + F(0.7152) * c[..., 1] + F(0.0722) * c[..., 2]


def _shift(a, dx, dy):
    """a[y + dy, x + dx] where that lies inside the frame (0 elsewhere), and the mask of where it does"""
    h, w = a.shape[:2]
    out, m = np.zeros_like(a), np.zeros((h, w), bool)
    ys, yd = slice(max(0, -dy), min(h, h - dy)), slice(max(0, dy), min(h, h + dy))
    xs, xd = slice(max(0, -dx), min(w, w - dx)), slice(max(0, dx), min(w, w + dx))
    out[ys, xs] = a[yd, xd]
    m[ys, xs] = True
    return out, m


B3 = {-2: 0.0625, -1: 0.25, 0: 0.375, 1: 0.25, 2: 0.0625}
G3 = {-1: 0.25, 0: 0.5, 1: 0.25}


def restated_level(col, ga, normal, obj, step, sigmas):
    """one à-trous level as denoise_rule.cuh states it, in float32 with the header's order of operations"""
    sc, sn, sz = (F(s) for s in sigmas)
    h, w = col.shape[:2]
    var = col[..., 3]
    vs, gs = np.zeros((h, w), F), np.zeros((h, w), F)
    for j in (-1, 0, 1):
        for i in (-1, 0, 1):
            v, m = _shift(var, i, j)
            g = F(G3[i] * G3[j])
            vs = np.where(m, vs + g * v, vs)
            gs = np.where(m, gs + g, gs)
    sd = np.sqrt(np.maximum(vs / gs, F(0)))
    z = ga[..., 3]
    x, y = np.arange(w), np.arange(h)
    xl, xr, yu, yd = np.maximum(x - 1, 0), np.minimum(x + 1, w - 1), np.maximum(y - 1, 0), np.minimum(y + 1, h - 1)
    gx = np.where(xr > xl, (z[:, xr] - z[:, xl]) / np.maximum(xr - xl, 1).astype(F), F(0))
    gy = np.where((yd > yu)[:, None], (z[yd, :] - z[yu, :]) / np.maximum(yd - yu, 1).astype(F)[:, None], F(0))
    lp = _lum(col)
    wsum, v2, acc = np.zeros((h, w), F), np.zeros((h, w), F), np.zeros((h, w, 3), F)
    for j in range(-2, 3):
        for i in range(-2, 3):
            cq, m = _shift(col, i * step, j * step)
            wt = np.full((h, w), F(B3[i] * B3[j]), F)
            if i or j:
                nq, _ = _shift(normal, i * step, j * step)
                oq, _ = _shift(obj, i * step, j * step)
                zq, _ = _shift(z, i * step, j * step)
                dz = np.abs(gx * F(i * step) + gy * F(j * step))
                nd = np.maximum(F(0), normal[..., 0] * nq[..., 0] + normal[..., 1] * nq[..., 1] + normal[..., 2] * nq[..., 2])
                wn = np.power(nd, sn)
                wz = np.exp(-np.abs(z - zq) / (sz * dz + F(1e-3)))
                wl = np.exp(-np.abs(lp - _lum(cq)) / (sc * sd + F(1e-4)))
                wt = wt * np.where(obj == oq, wn * wz * wl, F(0))
            wt = np.where(m, wt, F(0))
            wsum = wsum + wt
            acc = acc + wt[..., None] * cq[..., :3]
            v2 = v2 + wt * wt * cq[..., 3]
    inv = F(1) / wsum
    return np.concatenate([acc * inv[..., None], (v2 * inv * inv)[..., None]], axis=2)


def restated_filter(g, levels, sigmas=(4.0, 128.0, 1.0)):
    """rtb_denoise_image restated: demodulate, `levels` levels, remodulate (float32 [h, w, 3] linear colour)"""
    a = np.maximum(np.asarray(g["albedo"], F), F(1e-3))
    la = _lum(a)
    col = np.concatenate([np.asarray(g["color"], F) / a, (np.asarray(g["variance"], F) / (la * la))[..., None]], axis=2)
    ga = np.concatenate([np.asarray(g["albedo"], F), np.asarray(g["depth"], F)[..., None]], axis=2)
    for level in range(levels):
        col = restated_level(col, ga, np.asarray(g["normal"], F), np.asarray(g["obj"], np.int32), 1 << level, sigmas)
    return col[..., :3] * a


def random_guides(rng, h=37, w=53, n_obj=4):
    """piecewise-smooth random guides: a few objects in blobs, normals from a small palette plus noise, sloped depth"""
    yy, xx = np.mgrid[0:h, 0:w]
    obj = ((xx // 9 + yy // 7 + rng.integers(0, 2, (h, w))) % (n_obj + 1) - 1).astype(np.int32)   # -1 = miss
    pal = rng.normal(size=(n_obj + 1, 3))
    normal = pal[obj + 1] + 0.15 * rng.normal(size=(h, w, 3))
    normal /= np.linalg.norm(normal, axis=2, keepdims=True)
    normal[obj < 0] = 0.0
    depth = 50 + 0.3 * xx + 0.2 * yy + 5 * (obj + 1) + rng.normal(scale=0.05, size=(h, w))
    albedo = rng.uniform(0.05, 1.0, (n_obj + 1, 3))[obj + 1]
    albedo[obj < 0] = 1.0
    color = np.clip(albedo * rng.uniform(0.2, 0.9, (h, w, 1)) + rng.normal(scale=0.05, size=(h, w, 3)), 0, 1)
    variance = rng.uniform(0, 0.01, (h, w))
    return {k: v.astype(np.int32 if k == "obj" else F) for k, v in
            dict(color=color, variance=variance, albedo=albedo, normal=normal, depth=depth, obj=obj).items()}


@pytest.mark.parametrize("levels,sigmas", [(1, (4.0, 128.0, 1.0)), (2, (4.0, 128.0, 1.0)), (1, (0.5, 8.0, 0.2)), (3, (1e3, 0.0, 1e3))])
def test_atrous_matches_the_restated_rule(harness, levels, sigmas):
    g = random_guides(np.random.default_rng(3 + levels))
    got = harness(g, levels, sigmas)
    want = restated_filter(g, levels, sigmas)
    np.testing.assert_allclose(got, want, rtol=1e-6, atol=1e-6)
    assert np.abs(got - g["color"]).max() > 1e-3, "the filter changed nothing: the comparison checks nothing"


def test_constant_illumination_stays_constant(harness):
    g = random_guides(np.random.default_rng(11))
    illum = np.array([0.3, 0.5, 0.7], F)
    g["color"] = (illum * np.maximum(g["albedo"], F(1e-3))).astype(F)
    got = harness(g, 5)
    np.testing.assert_allclose(got, g["color"], rtol=1e-5, atol=1e-6)


def test_no_weight_crosses_object_ids(harness):
    # every object one flat colour, very different from its neighbours', permissive edge-stops otherwise: only the id can
    # keep the colours apart
    g = random_guides(np.random.default_rng(12))
    g["albedo"][:] = 1.0
    g["normal"][:] = np.array([0, 0, 1], F)
    g["depth"][:] = 10.0
    g["color"] = (np.array([[0.0, 0.0, 0.0], [1, 0, 0], [0, 1, 0], [0, 0, 1], [1, 1, 1]], F)[g["obj"] + 1]).astype(F)
    got = harness(g, 5, (1e6, 0.0, 1e6))
    np.testing.assert_allclose(got, g["color"], rtol=0, atol=1e-6)


def test_levels_zero_is_the_identity(harness):
    g = random_guides(np.random.default_rng(13))
    np.testing.assert_allclose(harness(g, 0), g["color"], rtol=1e-6, atol=1e-7)


# ---- server: "denoise": true ------------------------------------------------------------------------------------------
websockets = pytest.importorskip("websockets")


def test_denoise_request_reaches_the_factory(rtb):
    from test_adaptive_cpu import _Job, _send, _serve

    calls = []

    def factory(scene, spp, passes=1, **kw):
        calls.append((scene, spp, passes, kw))
        return _Job()

    port, stop = _serve(factory)
    try:
        for req in [{"spp": 64, "denoise": True}, {"spp": 64, "passes": 8, "denoise": True}, {"spp": 100, "noise": 2, "denoise": True},
                    {"spp": 64, "denoise": False}, {"spp": 64, "passes": 3}]:
            assert _send(port, {"type": "render", "scene": "cornell_box", **req}) == bytes([0, 1, 0, 0, 0, 0, 1, 2, 3])
    finally:
        stop()
    assert calls == [("cornell_box", 64, 1, {"denoise": True}), ("cornell_box", 64, 8, {"denoise": True}),
                     ("cornell_box", 96, 1, {"adaptive": {"target_levels": 2.0, "pass_spp": 16, "min_spp": 64}, "denoise": True}),
                     ("cornell_box", 64, 1, {}), ("cornell_box", 64, 3, {})]


@pytest.mark.parametrize("denoise", ["true", 1, 0, None, [True], {"levels": 5}])
def test_bad_denoise_closes_the_connection(rtb, denoise):
    from test_adaptive_cpu import _Job, _send, _serve

    calls = []
    port, stop = _serve(lambda *a, **kw: calls.append(a) or _Job())
    try:
        assert _send(port, {"type": "render", "scene": "cornell_box", "spp": 64, "denoise": denoise}, expect_close=True) == 1007
    finally:
        stop()
    assert calls == []
