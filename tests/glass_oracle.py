"""The f64 oracle with the dielectric material (tests/glass_oracle.cpp), for the glass parity tests.

oracle/oracle.py's OracleScene drives it: the C entry points and their signatures are the oracle's, so everything but the
scene parsing is inherited.  The library is compiled once per process (g++, the oracle Makefile's flags) into a temporary
directory, so the tree stays read-only.
"""
import ctypes as C
import math
import os
import subprocess
import tempfile
import threading

import numpy as np

from oracle import oracle as O

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "glass_oracle.cpp")
CXXFLAGS = ["-O3", "-march=x86-64-v3", "-ffp-contract=off", "-std=c++17", "-fPIC", "-pthread", "-shared"]
ACCEL_OCTREE_FAITHFUL, ACCEL_EXACT, EST_NEE, EST_MIS_DEAD = O.ACCEL_OCTREE_FAITHFUL, O.ACCEL_EXACT, O.EST_NEE, O.EST_MIS_DEAD

_lib = None
_mu = threading.Lock()


def lib():
    global _lib
    with _mu:
        if _lib is None:
            out = os.path.join(tempfile.mkdtemp(prefix="glass_oracle_"), "libglass_oracle.so")
            subprocess.run(["/usr/bin/g++", *CXXFLAGS, "-o", out, SRC], check=True, capture_output=True)
            L, ref = C.CDLL(out), O.lib()
            for name in dir(ref):   # the same entry points as the oracle's, with the same signatures
                if name.startswith("or_"):
                    f, g = getattr(L, name), getattr(ref, name)
                    f.argtypes, f.restype = g.argtypes, g.restype
            _lib = L
    return _lib


def _brdf(b, vec):
    """(kind, params) of a TOML brdf table, as or_add_object takes them"""
    bt = b["type"]
    if bt == "diffuse":
        return 0, vec(b["kd"])
    if bt == "specular":
        return 1, vec(b["ks"])
    if bt == "phong":
        if int(b["power"]) < 0:
            raise O.OracleError("parse: power must be usize")
        return 2, np.array([float(b["kd"]), float(b["ks"]), float(int(b["power"]))] + list(map(float, b["color_d"])) +
                           list(map(float, b["color_s"])))
    if bt == "dielectric":
        ior = float(b["ior"])
        tint = list(map(float, b.get("tint", [1.0, 1.0, 1.0])))
        if not (math.isfinite(ior) and ior > 0):
            raise O.OracleError("parse: dielectric ior must be finite and > 0")
        if len(tint) != 3 or not all(0.0 <= c <= 1.0 for c in tint):
            raise O.OracleError("parse: dielectric tint must be 3 numbers in [0, 1]")
        return 3, np.array([ior] + tint)
    raise O.OracleError(f"parse: unknown brdf type {bt}")


def _geometry(g, assets_dir):
    gt = g["type"]
    if gt == "sphere":
        return 0, np.array(list(map(float, g["pos"])) + [float(g["r"])]), b""
    if gt == "plane":
        return 1, np.array(list(map(float, g["pos"])) + list(map(float, g["n"]))), b""
    if gt == "mesh":
        if assets_dir is None:
            raise O.OracleError("mesh geometry needs assets_dir")
        return 2, np.zeros(6), os.path.join(assets_dir, g["path"]).encode()
    if gt == "cube":
        s = float(g["size"])
        return 3, np.array(list(map(float, g["pos"])) + [s, s, s]), b""
    if gt == "prism":
        return 3, np.array(list(map(float, g["pos"])) + list(map(float, g["size"]))), b""
    raise O.OracleError(f"parse: unknown geometry type {gt}")


TRANSFORMS = {"translate": 0, "scale": 1, "rotate_x": 2, "rotate_y": 3, "rotate_z": 4}


class OracleScene(O.OracleScene):
    """O.OracleScene on the glass oracle: the same parsing (tomllib, SceneSpec / to_scene) plus `type = "dielectric"`."""

    def __init__(self, spec: dict, assets_dir: str | None = None):
        self._f32, self._dt = False, np.float64
        L = self._L = lib()
        vec = lambda v: O._vec64(v)   # noqa: E731
        cam = spec["camera"]
        self._h = L.or_scene_new(O._dp(vec(cam["pos"])), O._dp(vec(cam["dir"])))
        self.spec = spec
        for ob in spec["objects"]:
            emitted = vec(ob.get("emitted", [0.0, 0.0, 0.0]))
            bk, bp = _brdf(ob["brdf"], vec)
            gk, gp, path = _geometry(ob["geometry"], assets_dir)
            kinds, vals = [], []
            for t in ob.get("transforms", []) or []:
                (k, v), = t.items()
                if k not in TRANSFORMS:
                    raise O.OracleError(f"parse: unknown transform {k}")
                kinds.append(TRANSFORMS[k])
                vals.append(list(map(float, v)) if k == "translate" else [float(v), 0.0, 0.0])
            ka = (C.c_int * max(1, len(kinds)))(*kinds)
            va = np.ascontiguousarray(np.array(vals, dtype=np.float64).reshape(-1)) if vals else np.zeros(3)
            rc = L.or_add_object(self._h, O._dp(emitted), bk, O._dp(np.ascontiguousarray(bp, dtype=np.float64)), gk,
                                 O._dp(np.ascontiguousarray(gp, dtype=np.float64)), path, len(kinds), ka, O._dp(va))
            if rc != 0:
                raise O.OracleError(L.or_last_error(self._h).decode())
        self.light_source = L.or_scene_finish(self._h)
        if self.light_source < 0:
            raise O.OracleError("no light source (reference: unreachable!() src/scene.rs:136)")
        self.set_modes(ACCEL_EXACT, EST_NEE)

    @classmethod
    def from_toml_string(cls, text: str, assets_dir: str | None = None) -> "OracleScene":
        import tomllib

        return cls(tomllib.loads(text), assets_dir)
