"""What a rough metal costs: k_shade MODE 6 (the general kernel with the dielectric and metal branches) against the kernels the
same scenes run without a metal, on one GPU, under EST_NEE.

Frames (seed 3, median of 3 timed renders after 2 warm-ups):
  * cornell_box at 600x450x64 and 1920x1080x256 as shipped (the mirror sphere, the fast kernels) and with the mirror sphere
    replaced by a roughness-0.3 metal of F0 = 1;
  * flying_unicorn at 1920x1080x64 as shipped and with Pegasus as rough gold (roughness 0.3, F0 = (1, 0.71, 0.29)).
Per frame: Msamples/s, rays per sample and wavefront iterations; k_shade / k_traverse ms (rtb_stats CUDA-event sums) come from
one more render with RTB_NO_GRAPH=1, because a frame that runs as CUDA graphs records no per-kernel events.  The card's name
and power limit are read in the same run.

usage: python tools/gpu_metal.py [out.json]   (the JSON result is always printed; out.json also receives it)"""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import raytracer_server_b200 as R
from gpu_adaptive import card
from gpu_lights import SEED, measure

SCENES = os.path.join(ROOT, "tests", "golden", "scenes")
MIRROR = 'brdf = { type = "specular", ks = [0.999, 0.999, 0.999] }'
PEGASUS = 'brdf = { type = "diffuse", kd = [0.9, 0.9, 0.9] }\ngeometry = { type = "mesh", path = "flying-unicorn.obj" }'


def pair(plain, metal, w, h, spp):
    return {"as shipped": measure(plain, w, h, spp, R.EST_NEE), "with the metal (MODE 6)": measure(metal, w, h, spp, R.EST_NEE)}


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else None
    res = {"card": card(), "seed": SEED, "estimator": "EST_NEE"}
    text = open(os.path.join(SCENES, "cornell_box.toml")).read()
    assert text.count(MIRROR) == 1
    cornell = R.Scene.from_toml_string(text)
    cornell_metal = R.Scene.from_toml_string(text.replace(MIRROR, 'brdf = { type = "metal", roughness = 0.3 }'))
    for w, h, spp in ((600, 450, 64), (1920, 1080, 256)):
        res[f"cornell_box {w}x{h}x{spp}, mirror sphere -> metal 0.3"] = pair(cornell, cornell_metal, w, h, spp)
        print(json.dumps(res[f"cornell_box {w}x{h}x{spp}, mirror sphere -> metal 0.3"]), flush=True)
    text = open(os.path.join(SCENES, "flying_unicorn.toml")).read()
    assert text.count(PEGASUS) == 1
    assets = os.path.join(SCENES, "assets")
    uni = R.Scene.from_toml_string(text, assets_dir=assets)
    gold = R.Scene.from_toml_string(text.replace(PEGASUS, PEGASUS.replace('type = "diffuse", kd = [0.9, 0.9, 0.9]',
                                                                          'type = "metal", roughness = 0.3, color = [1.0, 0.71, 0.29]')),
                                    assets_dir=assets)
    res["flying_unicorn 1920x1080x64, Pegasus -> rough gold 0.3"] = pair(uni, gold, 1920, 1080, 64)
    res["card_after"] = card()
    out = json.dumps(res, indent=1)
    print(out)
    if out_path:
        with open(out_path, "w") as f:
            f.write(out + "\n")


if __name__ == "__main__":
    main()
