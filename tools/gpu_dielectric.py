"""What glass costs: the dielectric material (brdf 3) against the mirror it replaces, on one GPU.

Frames (NEE, seed 3, median of 3 timed renders after 2 warm-ups):
  * glass Cornell box: cornell_box with object 7 turned into ior 1.5 glass at (73, 16.5, 78), smallpt's layout;
  * the mirror version of that box (object 7 a ks 0.999 mirror at the same place): the fast kernel (MODE 1), and the same
    under RTB_NO_FAST_SHADE=1 (the general kernel, MODE 0), which separates the cost of the dielectric branch from the cost
    of leaving the fast kernels;
  at 600x450x64 and 1920x1080x256;
  * flying_unicorn with Pegasus (object 6) as ior 1.5 glass at 1920x1080x64: every internal bounce is an LBVH query.
Per frame: Msamples/s, rays per sample and wavefront iterations; k_shade / k_traverse ms (rtb_stats CUDA-event sums) come from
one more render with RTB_NO_GRAPH=1, because a frame that runs as CUDA graphs records no per-kernel events.  The
card's name and power limit are read in the same run.

usage: python tools/gpu_dielectric.py [out.json]   (the JSON result is always printed; out.json also receives it)"""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import raytracer_server_b200 as R
from gpu_adaptive import card

SCENES = os.path.join(ROOT, "tests", "golden", "scenes")
SEED = 3
MIRROR7 = 'brdf = { type = "specular", ks = [0.999, 0.999, 0.999] }\ngeometry = { type = "sphere", pos = [73.0, 16.5, 68.0], r = 16.5 }'


def cornell(kind):
    text = open(os.path.join(SCENES, "cornell_box.toml")).read()
    assert MIRROR7 in text
    brdf = ('{ type = "dielectric", ior = 1.5 }' if kind == "glass" else '{ type = "specular", ks = [0.999, 0.999, 0.999] }')
    return text.replace(MIRROR7, f'brdf = {brdf}\ngeometry = {{ type = "sphere", pos = [73.0, 16.5, 78.0], r = 16.5 }}')


def glass_unicorn():
    text = open(os.path.join(SCENES, "flying_unicorn.toml")).read()
    old = 'brdf = { type = "diffuse", kd = [0.9, 0.9, 0.9] }\ngeometry = { type = "mesh", path = "flying-unicorn.obj" }'
    assert old in text
    return text.replace(old, 'brdf = { type = "dielectric", ior = 1.5 }\ngeometry = { type = "mesh", path = "flying-unicorn.obj" }')


def measure(g, w, h, spp, reps=3, env=None):
    old = {k: os.environ.get(k) for k in (env or {})}
    os.environ.update(env or {})
    try:
        for _ in range(2):
            g.render(w, h, spp, seed=SEED)
        runs = []
        for _ in range(reps):
            g.render(w, h, spp, seed=SEED)
            runs.append(g.stats())
        # the kernel split: frames that run as CUDA graphs record no per-kernel events, so one more render without the graph
        os.environ["RTB_NO_GRAPH"] = "1"
        g.render(w, h, spp, seed=SEED)
        split = g.stats()
    finally:
        os.environ.pop("RTB_NO_GRAPH", None)
        for k, v in old.items():
            if v is None: os.environ.pop(k, None)
            else: os.environ[k] = v
    st = sorted(runs, key=lambda s: s["render_ms"])[len(runs) // 2]
    rays = st["rays_primary"] + st["rays_extension"] + st["rays_shadow"]
    return {"frame": f"{w}x{h}x{spp}", "msamples_per_s": round(st["samples"] / st["render_ms"] / 1e3, 2),
            "render_ms": [round(s["render_ms"], 2) for s in runs], "rays_per_sample": round(rays / st["samples"], 3),
            "iterations": int(st["iterations"]), "no_graph_render_ms": round(split["render_ms"], 2),
            "no_graph_k_shade_ms": round(split["shade_ms"], 2), "no_graph_k_traverse_ms": round(split["extend_ms"], 2)}


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else None
    res = {"card": card(), "seed": SEED, "estimator": "nee", "cornell": {}, "flying_unicorn_glass": None}
    glass = R.Scene.from_toml_string(cornell("glass"))
    mirror = R.Scene.from_toml_string(cornell("mirror"))
    for w, h, spp in ((600, 450, 64), (1920, 1080, 256)):
        res["cornell"][f"{w}x{h}x{spp}"] = {
            "glass (MODE 3)": measure(glass, w, h, spp),
            "mirror, fast kernel (MODE 1)": measure(mirror, w, h, spp),
            "mirror, general kernel (MODE 0, RTB_NO_FAST_SHADE=1)": measure(mirror, w, h, spp, env={"RTB_NO_FAST_SHADE": "1"}),
        }
        print(json.dumps(res["cornell"][f"{w}x{h}x{spp}"]), flush=True)
    uni = R.Scene.from_toml(os.path.join(SCENES, "flying_unicorn.toml"))
    uni_glass = R.Scene.from_toml_string(glass_unicorn(), assets_dir=os.path.join(SCENES, "assets"))
    res["flying_unicorn_glass"] = {"glass Pegasus (MODE 3)": measure(uni_glass, 1920, 1080, 64),
                                   "diffuse Pegasus (as shipped)": measure(uni, 1920, 1080, 64)}
    res["card_after"] = card()
    text = json.dumps(res, indent=1)
    print(text)
    if out_path:
        with open(out_path, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
