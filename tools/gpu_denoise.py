"""What the denoiser buys and costs: cornell_box, cubes and flying_unicorn at 600x450 (NEE, seed 13) against the committed
4096-spp goldens (f64 oracle, seed 7; the golden's own noise caps every PSNR).

Per scene: PSNR of the raw and the denoised frame (default options: 5 levels, sigma_color 4, sigma_normal 128, sigma_depth
1) at 4 / 16 / 64 / 256 / 1024 spp, and the raw spp that reaches the denoised PSNR at 16 and 64 spp (interpolated in
log2(spp) on a ladder of raw renders up to 4096 spp).  A small sweep of the edge-stops at 16 spp.  The device time of the
guides (k_gbuffer) and of every filter kernel at 600x450 and 1920x1080, from torch.profiler over many launches, next to
the filter's CUDA-event time as rtb_stats.resolve_ms reports it.  The progressive cornell_box job of bench.py's C5
(passes = spp = 4096: one sample per pixel per frame) with and without denoising: frames/s and time to 30 / 35 dB.

usage: python tools/gpu_denoise.py [out.json]   (the JSON result is always printed; out.json also receives it)"""
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import numpy as np

import raytracer_server_b200 as R
from gpu_adaptive import card, time_to_db, uniform_spp_for
from parity_metrics import compare_regions, psnr

W, H, SEED = 600, 450, 13
SPPS = (4, 16, 64, 256, 1024)
LADDER = (4, 16, 64, 256, 1024, 2048, 4096)
SWEEP = [dict(sigma_color=c, sigma_normal=n, sigma_depth=z) for c, n, z in
         [(4, 128, 1), (2, 128, 1), (8, 128, 1), (16, 128, 1), (4, 32, 1), (4, 128, 0.25), (4, 128, 4)]]
KERNELS = ("k_gbuffer", "k_denoise_prep", "k_atrous", "k_denoise_out")


def kernel_times(g, w, h, reps=50):
    """device ms per call of every denoiser kernel (torch.profiler, CUDA activities) and the mean rtb_stats.resolve_ms"""
    import torch
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.init()
    for _ in range(3):
        g.render(w, h, 4, seed=1, denoise=True)
    ev_ms = []
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            g.render(w, h, 4, seed=1, denoise=True)
            ev_ms.append(g.stats()["resolve_ms"])
    tot = {k: 0.0 for k in KERNELS}
    for e in prof.key_averages():
        for k in KERNELS:
            if k in e.key:
                tot[k] += e.device_time_total / 1e3   # us -> ms
    per_call = {k: round(v / reps, 4) for k, v in tot.items()}
    per_call["filter_ms_events"] = round(float(np.mean(ev_ms)), 4)
    return per_call


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else None
    res = {"card": card(), "frame": f"{W}x{H}", "seed": SEED, "estimator": "nee", "options": "levels 5, sigma_color 4, sigma_normal 128, sigma_depth 1",
           "golden": "tests/golden/converged/<scene>_nee_600x450_4096spp_seed7.npz", "scenes": {}}
    print(res["card"], flush=True)
    for name in ("cornell_box", "cubes", "flying_unicorn"):
        g = R.Scene.from_toml(os.path.join(ROOT, "tests", "golden", "scenes", name + ".toml"))
        gold = np.load(os.path.join(ROOT, "tests", "golden", "converged", f"{name}_nee_600x450_4096spp_seed7.npz"))["rgb8"]
        g.render(W, H, 64, seed=1, denoise=True)   # warm-up
        ladder = [(spp, psnr(g.render(W, H, spp, seed=SEED), gold)) for spp in LADDER]
        sc = {"raw_ladder_psnr": {s: round(p, 3) for s, p in ladder}, "spp": {}, "sweep_16spp": []}
        for spp in SPPS:
            raw = g.render(W, H, spp, seed=SEED)
            dn = g.render(W, H, spp, seed=SEED, denoise=True)
            p = psnr(dn, gold)
            sc["spp"][spp] = {"psnr_raw": round(psnr(raw, gold), 3), "psnr_denoised": round(p, 3),
                              "region_raw": round(float(compare_regions(raw, gold)[0]), 5),
                              "region_denoised": round(float(compare_regions(dn, gold)[0]), 5),
                              "raw_spp_same_psnr": uniform_spp_for(p, ladder)}
            print(name, spp, sc["spp"][spp], flush=True)
        for opts in SWEEP:
            dn = g.render(W, H, 16, seed=SEED, denoise=opts)
            sc["sweep_16spp"].append({**opts, "psnr": round(psnr(dn, gold), 3)})
        print(name, "sweep", sc["sweep_16spp"], flush=True)
        if name == "cornell_box":
            sc["kernel_ms_600x450"] = kernel_times(g, 600, 450)
            sc["kernel_ms_1920x1080"] = kernel_times(g, 1920, 1080)
            print(name, sc["kernel_ms_600x450"], sc["kernel_ms_1920x1080"], flush=True)
            for dn in (None, True):
                t = time_to_db(R.RenderJob(g, W, H, 4096, seed=SEED, passes=4096, denoise=dn), gold, every=0)
                t["frames_per_s"] = round(t["frames"] / (t["total_ms"] / 1e3), 1)
                sc["progressive_c5_denoised" if dn else "progressive_c5_raw"] = t
                print(name, "denoised" if dn else "raw", t, flush=True)
        res["scenes"][name] = sc
        g.close()
    if out_path:
        os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
        with open(out_path, "w") as fh:
            json.dump(res, fh, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
