"""Host-side mirror of the reference's render interface over the C ABI.

Names follow the reference: ``Scene.from_toml`` (src/scene.rs:143), ``sample_pixel``
(src/server.rs:320), ``RenderJob.run`` (src/server.rs:157), ``LoadTomlError`` variants
(src/scene.rs:350-355).  All arithmetic happens in librtb200.so on the GPU.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

import numpy as np

from . import _abi
from ._abi import ACCEL_LBVH, ACCEL_OCTREE_REFERENCE, EST_MIS_BALANCE, EST_MIS_DEAD, EST_NEE, EST_NEE_ALL_LIGHTS, Adaptive, Denoise, ObjectDesc, ObjectInfo, Params, SceneDesc, SceneInfo, Stats


class RtbError(RuntimeError):
    code = 0

    def __init__(self, code: int, msg: str):
        super().__init__(f"[{code}] {msg}")
        self.code = code


class LoadTomlError(RtbError):
    """LoadTomlError::{Io, Parse, MeshLoad} — `.kind` names the variant."""

    @property
    def kind(self) -> str:
        return {_abi.RTB_EIO: "Io", _abi.RTB_EPARSE: "Parse", _abi.RTB_EMESH: "MeshLoad",
                _abi.RTB_ENOLIGHT: "NoLight", _abi.RTB_EUNSUPPORTED: "Unsupported"}.get(self.code, "Other")


def _check(rc: int, load: bool = False):
    if rc < 0:
        err = _abi.last_error()
        if load and rc in (_abi.RTB_EIO, _abi.RTB_EPARSE, _abi.RTB_EMESH, _abi.RTB_ENOLIGHT, _abi.RTB_EUNSUPPORTED):
            raise LoadTomlError(rc, err)
        raise RtbError(rc, err)
    return rc


def make_params(width: int, height: int, spp: int, *, use_mis: bool = False, seed: int = 0, rank: int = 0, world: int = 1,
                pool_paths: int = 0, count_work: bool = False, tune_refill: int = 0, tune_steps: int = 0,
                bin_bits: int | None = None, bin_octant_major: bool = False, estimator: int | None = None,
                accel: int = 0) -> Params:
    """bin_bits: coherence binning of the LBVH rays — None = library default, 0 = off, 2..5 = cell bits per axis."""
    p = Params()
    p.width, p.height, p.spp = width, height, spp
    p.estimator = estimator if estimator is not None else (EST_MIS_DEAD if use_mis else EST_NEE)
    p.seed = seed
    p.rank, p.world, p.pool_paths = rank, world, pool_paths
    p.accel = accel
    p.tuning[0] = 1 if count_work else 0
    p.tuning[1] = tune_refill
    p.tuning[2] = tune_steps
    p.tuning[3] = (0 if bin_bits is None else (1 if bin_bits <= 0 else max(2, bin_bits))) + (256 if bin_octant_major else 0)
    return p


def make_adaptive(spp: int, *, target_levels: float, pass_spp: int = 16, min_spp: int | None = None) -> Adaptive:
    """rtb_adaptive for a budget of `spp` samples per pixel; min_spp None = 4 passes, clipped to the budget."""
    o = Adaptive()
    o.target_levels = target_levels
    o.pass_spp = pass_spp
    o.min_spp = min(4 * pass_spp, spp) if min_spp is None else min_spp
    o.reserved = 0
    return o


def make_denoise(levels: int = 5, *, sigma_color: float = 4.0, sigma_normal: float = 128.0, sigma_depth: float = 1.0) -> Denoise:
    """rtb_denoise: `levels` à-trous levels (0 = the resolve through the denoise path, no filtering) and the three edge-stops."""
    o = Denoise()
    o.levels = levels
    o.sigma_color, o.sigma_normal, o.sigma_depth = sigma_color, sigma_normal, sigma_depth
    return o


def _denoise_opts(denoise) -> Denoise | None:
    """None (no denoising) | True (the defaults) | dict of make_denoise keywords | a Denoise"""
    if denoise is None or denoise is False:
        return None
    if denoise is True:
        return make_denoise()
    if isinstance(denoise, dict):
        return make_denoise(**denoise)
    return denoise


class Scene:
    """A loaded scene living on one GPU (immutable; share it between threads)."""

    def __init__(self, handle: int, name: str = ""):
        self._h = C.c_void_p(handle)
        self.name = name

    @property
    def info(self) -> SceneInfo:
        """rtb_scene_get_info: counts, LBVH shape, and (once ACCEL_OCTREE_REFERENCE has been used) the octree tables' sizes"""
        info = SceneInfo()
        _check(_abi.lib().rtb_scene_get_info(self._h, C.byref(info)))
        return info

    # ---- Scene::from_toml ------------------------------------------------------------------
    @classmethod
    def from_toml(cls, path: str, assets_dir: str | None = None, device: int = 0) -> "Scene":
        h = C.c_void_p()
        rc = _abi.lib().rtb_scene_load_toml(os.fsencode(path), os.fsencode(assets_dir) if assets_dir else None, device,
                                            C.byref(h))
        _check(rc, load=True)
        return cls(h.value, os.path.splitext(os.path.basename(path))[0])

    @classmethod
    def from_toml_string(cls, text: str, assets_dir: str | None = None, device: int = 0, name: str = "") -> "Scene":
        h = C.c_void_p()
        rc = _abi.lib().rtb_scene_load_toml_string(text.encode(), os.fsencode(assets_dir) if assets_dir else None, device,
                                                   C.byref(h))
        _check(rc, load=True)
        return cls(h.value, name)

    @classmethod
    def from_objects(cls, camera_pos, camera_dir, objects: list, device: int = 0, name: str = "") -> "Scene":
        """Programmatic scene (rtb_scene_create).  Each object is a dict: emitted (opt), brdf = ("diffuse", kd) |
        ("specular", ks) | ("phong", kd, ks, power, color_d, color_s) | ("dielectric", ior, tint) (tint optional, default
        (1, 1, 1)), geometry = ("sphere", pos, r) | ("plane", pos, n) | ("mesh", triangles[n, 3, 3])."""
        arr = (ObjectDesc * max(1, len(objects)))()
        keep = []
        for d, ob in zip(arr, objects):
            d.emitted[:] = list(map(float, ob.get("emitted", (0.0, 0.0, 0.0))))
            b = ob["brdf"]
            d.brdf = {"diffuse": 0, "specular": 1, "phong": 2, "dielectric": 3}[b[0]]
            if b[0] == "dielectric":
                d.k[:] = [float(b[1]), 0.0, 0.0]
                d.color_d[:] = list(map(float, b[2])) if len(b) > 2 else [1.0, 1.0, 1.0]
            elif b[0] == "phong":
                d.k[:] = [float(b[1]), float(b[2]), float(b[3])]
                d.color_d[:] = list(map(float, b[4]))
                d.color_s[:] = list(map(float, b[5]))
            else:
                d.k[:] = list(map(float, b[1]))
            g = ob["geometry"]
            d.geometry = {"sphere": 0, "plane": 1, "mesh": 2}[g[0]]
            if g[0] == "sphere":
                d.pos[:] = list(map(float, g[1]))
                d.r = float(g[2])
            elif g[0] == "plane":
                d.pos[:] = list(map(float, g[1]))
                d.n[:] = list(map(float, g[2]))
            else:
                tri = np.ascontiguousarray(g[1], dtype=np.float32).reshape(-1, 9)
                keep.append(tri)
                d.triangles = tri.ctypes.data_as(C.POINTER(C.c_float))
                d.n_triangles = tri.shape[0]
        desc = SceneDesc()
        desc.camera_pos[:] = list(map(float, camera_pos))
        desc.camera_dir[:] = list(map(float, camera_dir))
        desc.n_objects = len(objects)
        desc.objects = arr
        h = C.c_void_p()
        _check(_abi.lib().rtb_scene_create(C.byref(desc), device, C.byref(h)), load=True)
        return cls(h.value, name)

    # ---- scene + BVH as one blob (multi-GPU broadcast) ---------------------------------------------
    def export(self) -> np.ndarray:
        """rtb_scene_export: the loaded objects and the device-built LBVH tables as one uint8 array."""
        n = _abi.lib().rtb_scene_export(self._h, None, 0)
        _check(int(n))
        buf = np.empty(int(n), dtype=np.uint8)
        _check(int(_abi.lib().rtb_scene_export(self._h, buf.ctypes.data_as(C.c_void_p), buf.size)))
        return buf

    @classmethod
    def from_export(cls, blob, device: int = 0, name: str = "") -> "Scene":
        """rtb_scene_import: a scene handle on `device` from another handle's export — no parsing, no BVH build."""
        blob = np.ascontiguousarray(blob, dtype=np.uint8)
        h = C.c_void_p()
        _check(_abi.lib().rtb_scene_import(blob.ctypes.data_as(C.c_void_p), blob.size, device, C.byref(h)), load=True)
        return cls(h.value, name)

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            _abi.lib().rtb_scene_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def light_source(self) -> int:
        return self.info.light_object

    def object(self, index: int) -> dict:
        o = ObjectInfo()
        _check(_abi.lib().rtb_scene_object(self._h, index, C.byref(o)))
        d = {}
        for name, typ in o._fields_:
            v = getattr(o, name)
            d[name] = list(v) if hasattr(v, "__len__") else v
        return d

    def triangles(self) -> np.ndarray:
        n = _abi.lib().rtb_scene_triangles(self._h, None, 0)
        out = np.zeros((max(n, 0), 3, 3), dtype=np.float32)
        if n > 0:
            _abi.lib().rtb_scene_triangles(self._h, out.ctypes.data_as(C.POINTER(C.c_float)), n)
        return out

    def lights(self) -> dict:
        """The light table of EST_NEE_ALL_LIGHTS (rtb_scene_lights): object index int32 [n], selection probability and area
        float64 [n], in object order."""
        L = _abi.lib()
        n = _check(int(L.rtb_scene_lights(self._h, None, None, None, 0)))
        obj, prob, area = np.zeros(n, np.int32), np.zeros(n, np.float64), np.zeros(n, np.float64)
        dp = C.POINTER(C.c_double)
        L.rtb_scene_lights(self._h, obj.ctypes.data_as(C.POINTER(C.c_int32)), prob.ctypes.data_as(dp), area.ctypes.data_as(dp), n)
        return {"objects": obj, "prob": prob, "area": area}

    def octree_stats(self, index: int) -> dict:
        """Octree::build for mesh object `index` on the host (what ACCEL_OCTREE_REFERENCE traverses)."""
        c = (C.c_int64 * 4)()
        _check(_abi.lib().rtb_scene_octree_stats(self._h, index, c))
        return {"nodes": c[0], "parents": c[1], "leaves": c[2], "tri_refs": c[3]}

    def upload(self) -> int:
        b = C.c_uint64()
        _check(_abi.lib().rtb_scene_upload(self._h, C.byref(b)))
        return b.value

    def stats(self) -> dict:
        s = Stats()
        _check(_abi.lib().rtb_get_stats(self._h, C.byref(s)))
        return s.as_dict()

    # ---- RenderJob::run, blocking whole-frame form ----------------------------------------------
    def render(self, width: int, height: int, spp: int, *, use_mis: bool = False, seed: int = 0, rank: int = 0,
               world: int = 1, pool_paths: int = 0, out: np.ndarray | None = None, count_work: bool = False,
               tune_refill: int = 0, tune_steps: int = 0, bin_bits: int | None = None, bin_octant_major: bool = False,
               estimator: int | None = None, accel: int = 0, denoise=None) -> np.ndarray:
        """Returns the frame as uint8 [height, width, 3], row 0 = top (the bytes of src/server.rs:187-189).
        denoise: None = rtb_render; True / dict of make_denoise keywords / Denoise = rtb_render_denoised (whole frames)."""
        p = make_params(width, height, spp, use_mis=use_mis, seed=seed, rank=rank, world=world, pool_paths=pool_paths,
                        count_work=count_work, tune_refill=tune_refill, tune_steps=tune_steps, bin_bits=bin_bits,
                        bin_octant_major=bin_octant_major, estimator=estimator, accel=accel)
        if out is None:
            out = np.zeros((height, width, 3), dtype=np.uint8)
        assert out.dtype == np.uint8 and out.flags["C_CONTIGUOUS"] and out.size == width * height * 3
        dn = _denoise_opts(denoise)
        if dn is not None:
            _check(_abi.lib().rtb_render_denoised(self._h, C.byref(p), None, C.byref(dn), out.ctypes.data_as(C.POINTER(C.c_uint8)),
                                                  None, None, None))
        else:
            _check(_abi.lib().rtb_render(self._h, C.byref(p), out.ctypes.data_as(C.POINTER(C.c_uint8)), None))
        return out

    def render_adaptive(self, width: int, height: int, spp: int, *, target_levels: float, pass_spp: int = 16,
                        min_spp: int | None = None, use_mis: bool = False, seed: int = 0, accel: int = 0, denoise=None):
        """Adaptive sampling (rtb_render_adaptive): spp is the budget; each 32x32 tile stops once every pixel's estimated
        standard error is <= target_levels 8-bit output levels.  Returns (frame uint8 [h, w, 3], tile_spp int32 [ty, tx],
        tile_error float32 [ty, tx]).  denoise as for render (rtb_render_denoised)."""
        p = make_params(width, height, spp, use_mis=use_mis, seed=seed, accel=accel)
        o = make_adaptive(spp, target_levels=target_levels, pass_spp=pass_spp, min_spp=min_spp)
        ty, tx = (height + 31) // 32, (width + 31) // 32
        out = np.zeros((height, width, 3), dtype=np.uint8)
        tile_spp = np.zeros((ty, tx), dtype=np.int32)
        tile_error = np.zeros((ty, tx), dtype=np.float32)
        args = (out.ctypes.data_as(C.POINTER(C.c_uint8)), tile_spp.ctypes.data_as(C.POINTER(C.c_int32)),
                tile_error.ctypes.data_as(C.POINTER(C.c_float)), None)
        dn = _denoise_opts(denoise)
        if dn is not None:
            _check(_abi.lib().rtb_render_denoised(self._h, C.byref(p), C.byref(o), C.byref(dn), *args))
        else:
            _check(_abi.lib().rtb_render_adaptive(self._h, C.byref(p), C.byref(o), *args))
        return out, tile_spp, tile_error

    def gbuffer(self, width: int, height: int, accel: int = 0) -> dict:
        """The denoiser's guides (rtb_scene_gbuffer): albedo float32 [h, w, 3], normal float32 [h, w, 3], depth float32
        [h, w], obj int32 [h, w] (-1 = miss); row 0 = top."""
        albedo = np.empty((height, width, 3), dtype=np.float32)
        normal = np.empty((height, width, 3), dtype=np.float32)
        depth = np.empty((height, width), dtype=np.float32)
        obj = np.empty((height, width), dtype=np.int32)
        fp = C.POINTER(C.c_float)
        _check(_abi.lib().rtb_scene_gbuffer(self._h, width, height, accel, albedo.ctypes.data_as(fp), normal.ctypes.data_as(fp),
                                            depth.ctypes.data_as(fp), obj.ctypes.data_as(C.POINTER(C.c_int32))))
        return {"albedo": albedo, "normal": normal, "depth": depth, "obj": obj}

    def render_device(self, params: Params, d_rgb8_tiles: int, d_subpixel_sums: int = 0) -> int:
        """Device-resident render: raw device pointers (e.g. torch tensor .data_ptr())."""
        return _check(_abi.lib().rtb_render_device(self._h, C.byref(params), C.c_void_p(d_rgb8_tiles),
                                                   C.c_void_p(d_subpixel_sums) if d_subpixel_sums else None, None))

    # ---- parity hooks -----------------------------------------------------------------------------
    def trace_primary(self, width: int, height: int, sx: int = 0, sy: int = 0, dx: float = 0.0, dy: float = 0.0):
        n = width * height
        obj = np.empty(n, dtype=np.int32)
        tri = np.empty(n, dtype=np.int32)
        t = np.empty(n, dtype=np.float32)
        ip, fp = C.POINTER(C.c_int32), C.POINTER(C.c_float)
        _check(_abi.lib().rtb_trace_primary(self._h, width, height, sx, sy, dx, dy, obj.ctypes.data_as(ip),
                                            tri.ctypes.data_as(ip), t.ctypes.data_as(fp)))
        return {"obj": obj, "tri": tri, "t": t}

    def trace_rays(self, org, dirs, count_work: bool = False, accel: int = 0):
        org = np.ascontiguousarray(org, dtype=np.float32).reshape(-1, 3)
        dirs = np.ascontiguousarray(dirs, dtype=np.float32).reshape(-1, 3)
        n = org.shape[0]
        obj = np.empty(n, dtype=np.int32)
        tri = np.empty(n, dtype=np.int32)
        t = np.empty(n, dtype=np.float32)
        work = (C.c_uint64 * 2)(0, 0)
        ip, fp = C.POINTER(C.c_int32), C.POINTER(C.c_float)
        if accel:
            _check(_abi.lib().rtb_trace_rays_accel(self._h, accel, n, org.ctypes.data_as(fp), dirs.ctypes.data_as(fp), obj.ctypes.data_as(ip),
                                                   tri.ctypes.data_as(ip), t.ctypes.data_as(fp)))
        else:
            _check(_abi.lib().rtb_trace_rays(self._h, n, org.ctypes.data_as(fp), dirs.ctypes.data_as(fp), obj.ctypes.data_as(ip),
                                             tri.ctypes.data_as(ip), t.ctypes.data_as(fp), work if count_work else None))
        res = {"obj": obj, "tri": tri, "t": t}
        if count_work:
            res["work"] = {"node_visits": work[0], "tri_tests": work[1]}
        return res

    def sample_radiance(self, width, height, spp, px, py, sample_idx, *, use_mis=False, seed=0, estimator=None, accel=0) -> np.ndarray:
        p = make_params(width, height, spp, use_mis=use_mis, seed=seed, estimator=estimator, accel=accel)
        px = np.ascontiguousarray(px, dtype=np.int32)
        py = np.ascontiguousarray(py, dtype=np.int32)
        si = np.ascontiguousarray(sample_idx, dtype=np.int32)
        out = np.empty((px.size, 3), dtype=np.float32)
        ip = C.POINTER(C.c_int32)
        _check(_abi.lib().rtb_sample_radiance(self._h, C.byref(p), px.size, px.ctypes.data_as(ip), py.ctypes.data_as(ip),
                                              si.ctypes.data_as(ip), out.ctypes.data_as(C.POINTER(C.c_float))))
        return out


def sample_pixels(xs, ys_screen, width: int, height: int, samples_per_pixel: int, scene: Scene, *, seed: int = 0,
                  use_mis: bool = False, estimator: int | None = None) -> np.ndarray:
    """sample_pixel for a batch of pixels (x, screen row y; rtb_sample_pixels): float32 [n, 3], the Vec3 of
    src/server.rs:363 per pixel (0..255.5; `as u8` truncates it to the frame's bytes)."""
    p = make_params(width, height, samples_per_pixel, use_mis=use_mis, seed=seed, estimator=estimator)
    px = np.ascontiguousarray(xs, dtype=np.int32).reshape(-1)
    py = np.ascontiguousarray(ys_screen, dtype=np.int32).reshape(-1)
    assert px.size == py.size
    out = np.empty((px.size, 3), dtype=np.float32)
    ip = C.POINTER(C.c_int32)
    _check(_abi.lib().rtb_sample_pixels(scene._h, C.byref(p), px.size, px.ctypes.data_as(ip), py.ctypes.data_as(ip),
                                        out.ctypes.data_as(C.POINTER(C.c_float))))
    return out


def sample_pixel(x: int, y: int, width: int, height: int, samples_per_pixel: int, scene: Scene, *, seed: int = 0,
                 use_mis: bool = False) -> np.ndarray:
    """src/server.rs:320-364 for ONE pixel, same arguments: y is the sampler's own bottom-up row (the caller passes
    height - y_screen - 1, src/server.rs:181).  Returns the Vec3 (0..255.5) — only this pixel's paths are traced."""
    return sample_pixels([x], [height - y - 1], width, height, samples_per_pixel, scene, seed=seed, use_mis=use_mis)[0]


class RenderJob:
    """The streaming form of RenderJob::run: yields (x, y, rgb[n,3]) records, 60 pixels at most,
    rows top-down — the payload of the reference's binary messages (src/server.rs:173-190)."""

    PIXELS_PER_MSG = 60

    def __init__(self, scene: Scene, width: int, height: int, samples_per_pixel: int, *, passes: int = 1, seed: int = 0,
                 use_mis: bool = False, pool_paths: int = 0, accel: int = 0, adaptive: dict | None = None, denoise=None,
                 estimator: int | None = None):
        """adaptive: dict(target_levels=..., pass_spp=16, min_spp=None) makes this an adaptive job (rtb_job_begin_adaptive):
        samples_per_pixel is the budget, `passes` is ignored and the job re-sends the frame once per pass until every tile
        has converged.  denoise (True / dict of make_denoise keywords / Denoise): every frame the job sends is denoised
        (rtb_job_begin_denoised); a single-pass job then renders the frame as one band.  estimator: an EST_* constant
        (None = EST_MIS_DEAD if use_mis else EST_NEE)."""
        self.scene = scene
        self.params = make_params(width, height, samples_per_pixel, use_mis=use_mis, seed=seed, pool_paths=pool_paths, accel=accel,
                                  estimator=estimator)
        self._h = C.c_void_p()
        # guards the handle: stop() may come from another thread (the server's event loop) while close() frees the job
        self._lock = threading.Lock()
        dn = _denoise_opts(denoise)
        if dn is not None:
            self.adaptive = make_adaptive(samples_per_pixel, **adaptive) if adaptive is not None else None
            self.denoise = dn
            _check(_abi.lib().rtb_job_begin_denoised(scene._h, C.byref(self.params), passes,
                                                     C.byref(self.adaptive) if self.adaptive is not None else None, C.byref(dn),
                                                     C.byref(self._h)))
        elif adaptive is not None:
            self.adaptive = make_adaptive(samples_per_pixel, **adaptive)
            _check(_abi.lib().rtb_job_begin_adaptive(scene._h, C.byref(self.params), C.byref(self.adaptive), C.byref(self._h)))
        else:
            _check(_abi.lib().rtb_job_begin(scene._h, C.byref(self.params), passes, C.byref(self._h)))
        self._buf = (C.c_uint8 * (256 * (6 + 3 * self.PIXELS_PER_MSG)))()
        self.cancelled = False
        self.final_stats = None

    def messages(self, max_records: int = 256):
        """Iterates over byte strings, each one reference wire message (header + n*rgb)."""
        L = _abi.lib()
        nbytes = C.c_int64()
        while True:
            rc = L.rtb_job_next_messages(self._h, self._buf, len(self._buf), min(max_records, 256), C.byref(nbytes))
            if rc == _abi.RTB_ESTOPPED:
                self.cancelled = True
                return
            _check(rc)
            if rc == 0 and nbytes.value == 0:
                return
            raw = bytes(self._buf[: nbytes.value])
            off = 0
            while off < len(raw):
                n = raw[off + 1]
                yield raw[off: off + 6 + 3 * n]
                off += 6 + 3 * n

    def frames(self):
        """Progressive display: yields (pass_index, frame uint8 [h, w, 3]) once per finished pass."""
        L = _abi.lib()
        h, w = self.params.height, self.params.width
        idx = C.c_int32()
        while True:
            frame = np.empty((h, w, 3), dtype=np.uint8)
            rc = L.rtb_job_next_frame(self._h, frame.ctypes.data_as(C.POINTER(C.c_uint8)), C.byref(idx))
            if rc == _abi.RTB_ESTOPPED:
                self.cancelled = True
                return
            _check(rc)
            if rc == 0:
                return
            yield idx.value, frame

    def stats(self) -> dict:
        """Counters of the job so far (rtb_job_stats), incl. first_record_ms / wall_ms; after close(): the final ones."""
        with self._lock:
            if not self._h.value:
                return dict(self.final_stats or {})
            s = Stats()
            _check(_abi.lib().rtb_job_stats(self._h, C.byref(s)))
            return s.as_dict()

    def stop(self):
        with self._lock:   # never touches a handle close() has already handed to rtb_job_end
            if self._h.value:
                _abi.lib().rtb_job_cancel(self._h)

    def close(self) -> bool:
        """Returns True if the job was stopped before completion (RenderJob::run's bool)."""
        with self._lock:
            h, self._h = self._h, C.c_void_p()   # from here on stop() / stats() see no handle
            if h.value:
                s = Stats()
                if _abi.lib().rtb_job_stats(h, C.byref(s)) == 0:
                    self.final_stats = s.as_dict()
        if not h.value:
            return self.cancelled
        # rtb_job_end joins the worker threads: outside the lock, so that a concurrent stop() returns at once (no handle)
        # -- a stop() that raced ahead of the swap has already cancelled the job, which only makes the join faster
        rc = _abi.lib().rtb_job_end(h)
        self.cancelled = self.cancelled or rc == _abi.RTB_ECANCELLED
        return self.cancelled

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def denoise_image(color, variance, albedo, normal, depth, obj, *, levels: int = 5, sigma_color: float = 4.0,
                  sigma_normal: float = 128.0, sigma_depth: float = 1.0, device: int = 0) -> np.ndarray:
    """The filter alone (rtb_denoise_image) on host arrays: color / albedo / normal [h, w, 3], variance / depth [h, w] float,
    obj [h, w] int.  Returns the denoised linear colour float32 [h, w, 3] (before clamp and gamma)."""
    color = np.ascontiguousarray(color, dtype=np.float32)
    h, w = color.shape[:2]
    arrs = [np.ascontiguousarray(a, dtype=np.float32) for a in (variance, albedo, normal, depth)]
    obj = np.ascontiguousarray(obj, dtype=np.int32)
    assert color.shape == (h, w, 3) and arrs[1].shape == arrs[2].shape == (h, w, 3)
    assert arrs[0].shape == arrs[3].shape == obj.shape == (h, w)
    out = np.empty((h, w, 3), dtype=np.float32)
    o = make_denoise(levels, sigma_color=sigma_color, sigma_normal=sigma_normal, sigma_depth=sigma_depth)
    fp = C.POINTER(C.c_float)
    _check(_abi.lib().rtb_denoise_image(device, w, h, C.byref(o), color.ctypes.data_as(fp), *[a.ctypes.data_as(fp) for a in arrs],
                                        obj.ctypes.data_as(C.POINTER(C.c_int32)), out.ctypes.data_as(fp)))
    return out


def fp32_peak_tflops(device: int = 0) -> float:
    v = C.c_double()
    _check(_abi.lib().rtb_fp32_peak(device, C.byref(v)))
    return v.value
