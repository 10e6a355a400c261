"""What next-event estimation over every emitter costs: EST_NEE_ALL_LIGHTS (k_shade MODE 4) against EST_NEE, on one GPU.

Frames (seed 3, median of 3 timed renders after 2 warm-ups):
  * cornell_box at 600x450x64 and 1920x1080x256, flying_unicorn at 1920x1080x64: one sphere light, where both estimators give
    the same image, so the difference is the price of the general kernel and the table lookup;
  * a two-light Cornell box (cornell_box plus a bluish sphere light of radius 6 at (20, 60, 60)) at 600x450x64: throughput, and
    the mean Rec. 709 luminance of both 8-bit images — the light estimator 0 leaves out.
Per frame: Msamples/s, rays per sample and wavefront iterations; k_shade / k_traverse ms (rtb_stats CUDA-event sums) come from
one more render with RTB_NO_GRAPH=1, because a frame that runs as CUDA graphs records no per-kernel events.  The card's name
and power limit are read in the same run.

usage: python tools/gpu_lights.py [out.json]   (the JSON result is always printed; out.json also receives it)"""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import raytracer_server_b200 as R
from gpu_adaptive import card

SCENES = os.path.join(ROOT, "tests", "golden", "scenes")
SEED = 3
LIGHT_B = """
[[objects]]
emitted = [6.0, 12.0, 30.0]
brdf = { type = "diffuse", kd = [0.0, 0.0, 0.0] }
geometry = { type = "sphere", pos = [20.0, 60.0, 60.0], r = 6.0 }
"""
LUM = np.array([0.2126, 0.7152, 0.0722])


def measure(g, w, h, spp, estimator, reps=3):
    for _ in range(2):
        g.render(w, h, spp, seed=SEED, estimator=estimator)
    runs = []
    for _ in range(reps):
        frame = g.render(w, h, spp, seed=SEED, estimator=estimator)
        runs.append(g.stats())
    os.environ["RTB_NO_GRAPH"] = "1"   # the kernel split: frames that run as CUDA graphs record no per-kernel events
    try:
        g.render(w, h, spp, seed=SEED, estimator=estimator)
        split = g.stats()
    finally:
        os.environ.pop("RTB_NO_GRAPH", None)
    st = sorted(runs, key=lambda s: s["render_ms"])[len(runs) // 2]
    rays = st["rays_primary"] + st["rays_extension"] + st["rays_shadow"]
    return {"frame": f"{w}x{h}x{spp}", "msamples_per_s": round(st["samples"] / st["render_ms"] / 1e3, 2),
            "render_ms": [round(s["render_ms"], 2) for s in runs], "rays_per_sample": round(rays / st["samples"], 3),
            "iterations": int(st["iterations"]), "no_graph_render_ms": round(split["render_ms"], 2),
            "no_graph_k_shade_ms": round(split["shade_ms"], 2), "no_graph_k_traverse_ms": round(split["extend_ms"], 2),
            "mean_luminance_8bit": round(float((frame.reshape(-1, 3).astype(np.float64) @ LUM).mean()), 3)}


def pair(g, w, h, spp):
    return {"EST_NEE (estimator 0)": measure(g, w, h, spp, R.EST_NEE),
            "EST_NEE_ALL_LIGHTS (estimator 3, MODE 4)": measure(g, w, h, spp, R.EST_NEE_ALL_LIGHTS)}


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else None
    res = {"card": card(), "seed": SEED, "single_light": {}, "two_light_cornell": None}
    cornell = R.Scene.from_toml(os.path.join(SCENES, "cornell_box.toml"))
    for w, h, spp in ((600, 450, 64), (1920, 1080, 256)):
        res["single_light"][f"cornell_box {w}x{h}x{spp}"] = pair(cornell, w, h, spp)
        print(json.dumps(res["single_light"][f"cornell_box {w}x{h}x{spp}"]), flush=True)
    uni = R.Scene.from_toml(os.path.join(SCENES, "flying_unicorn.toml"))
    res["single_light"]["flying_unicorn 1920x1080x64"] = pair(uni, 1920, 1080, 64)
    two = R.Scene.from_toml_string(open(os.path.join(SCENES, "cornell_box.toml")).read() + LIGHT_B)
    p = pair(two, 600, 450, 64)
    e0, e3 = (p[k]["mean_luminance_8bit"] for k in p)
    res["two_light_cornell"] = {**p, "mean_luminance_missing_under_estimator_0": round(e3 - e0, 3)}
    res["card_after"] = card()
    text = json.dumps(res, indent=1)
    print(text)
    if out_path:
        with open(out_path, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
