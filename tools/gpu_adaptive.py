"""What adaptive sampling saves: cornell_box, cubes and flying_unicorn at 600x450 with a budget of 4096 spp, against the
committed 4096-spp goldens (f64 oracle, seed 7; renders here use seed 11, so the golden's own noise caps every PSNR).

Per scene: the uniform rtb_render at 4096 spp and render_adaptive at targets 0.5 / 1 / 2 levels (pass_spp 16, min_spp 64):
samples spent, wall ms, PSNR and per-channel MRE against the golden, and the uniform spp that reaches the same PSNR
(interpolated in log2(spp) on a ladder of uniform renders).  cornell_box also gets the time to 30 / 35 dB of an adaptive
job against the uniform progressive job of bench.py's C5 (passes = spp = 4096: one sample per pixel per frame).

usage: python tools/gpu_adaptive.py [out.json]   (the JSON result is always printed; out.json also receives it)"""
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np

import raytracer_server_b200 as R
from parity_metrics import channel_mre, psnr

W, H, BUDGET, SEED = 600, 450, 4096, 11
TARGETS = (0.5, 1.0, 2.0)
LADDER = (64, 128, 256, 512, 1024, 2048, 4096)
DB_MARKS = (30, 35)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown (nvidia-smi failed)"


def timed(fn):
    t0 = time.perf_counter()
    r = fn()
    return r, (time.perf_counter() - t0) * 1e3


def uniform_spp_for(p, ladder):
    """uniform spp at which the ladder's PSNR reaches p (linear in log2 spp between rungs)"""
    spps = np.array([s for s, _ in ladder], dtype=np.float64)
    ps = np.array([q for _, q in ladder])
    if p <= ps[0]:
        return f"<= {int(spps[0])}"
    if p > ps[-1]:
        return f"> {int(spps[-1])}"
    k = int(np.nonzero(ps >= p)[0][0])
    f = (p - ps[k - 1]) / (ps[k] - ps[k - 1])
    return round(float(2 ** (np.log2(spps[k - 1]) + f * (np.log2(spps[k]) - np.log2(spps[k - 1])))), 1)


def time_to_db(job, gold, every=1):
    """(frames, {db: {frames, ms}}) of a job; frames are kept (on a schedule) and scored after the job, so the PSNR
    bookkeeping does not slow the consumer"""
    kept, n, nxt = [], 0, 1
    t0 = time.perf_counter()
    for _, f in job.frames():
        n += 1
        if every == 1 or n >= nxt:
            kept.append((n, (time.perf_counter() - t0) * 1e3, f))
            nxt = max(n + 1, int(n * 1.25))
    total_ms = (time.perf_counter() - t0) * 1e3
    job.close()
    reached = {db: None for db in DB_MARKS}
    for n_, ms, f in kept:
        p = psnr(f, gold)
        for db in DB_MARKS:
            if reached[db] is None and p >= db:
                reached[db] = {"frames": n_, "ms": round(ms, 1)}
    return {"frames": n, "total_ms": round(total_ms, 1), "final_psnr": round(psnr(kept[-1][2], gold), 3), "time_to_psnr_db": reached}


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else None
    res = {"card": card(), "frame": f"{W}x{H}", "budget_spp": BUDGET, "seed": SEED, "pass_spp": 16, "min_spp": 64,
           "golden": "tests/golden/converged/<scene>_nee_600x450_4096spp_seed7.npz", "scenes": {}}
    print(res["card"], flush=True)
    for name in ("cornell_box", "cubes", "flying_unicorn"):
        g = R.Scene.from_toml(os.path.join(ROOT, "tests", "golden", "scenes", name + ".toml"))
        gold = np.load(os.path.join(ROOT, "tests", "golden", "converged", f"{name}_nee_600x450_4096spp_seed7.npz"))["rgb8"]
        g.render(W, H, 64, seed=1)                                                    # warm-up
        g.render_adaptive(W, H, 256, target_levels=2.0, seed=1)
        ladder = []
        for spp in LADDER:
            f, ms = timed(lambda: g.render(W, H, spp, seed=SEED))
            ladder.append((spp, psnr(f, gold)))
            if spp == BUDGET:
                uni = {"samples": g.stats()["samples"], "wall_ms": round(ms, 1), "psnr": round(ladder[-1][1], 3),
                       "channel_mre": [round(float(v), 5) for v in channel_mre(f, gold)]}
        sc = {"uniform_4096": uni, "uniform_ladder_psnr": {s: round(p, 3) for s, p in ladder}, "adaptive": {}}
        for target in TARGETS:
            (f, tile_spp, _), ms = timed(lambda: g.render_adaptive(W, H, BUDGET, target_levels=target, pass_spp=16, min_spp=64, seed=SEED))
            st = g.stats()
            p = psnr(f, gold)
            sc["adaptive"][str(target)] = {
                "samples": st["samples"], "samples_vs_uniform": round(st["samples"] / uni["samples"], 4), "wall_ms": round(ms, 1),
                "mean_spp": round(st["samples"] / (W * H), 1), "psnr": round(p, 3), "channel_mre": [round(float(v), 5) for v in channel_mre(f, gold)],
                "uniform_spp_same_psnr": uniform_spp_for(p, ladder), "tiles_at_budget": int((tile_spp == BUDGET).sum()), "tiles": int(tile_spp.size),
                "iterations": st["iterations"], "kernel_launches": st["kernel_launches"]}
            print(name, target, sc["adaptive"][str(target)], flush=True)
        if name == "cornell_box":
            sc["time_to_db_uniform_progressive_c5"] = time_to_db(R.RenderJob(g, W, H, BUDGET, seed=SEED, passes=BUDGET), gold, every=0)
            for target in TARGETS:
                sc[f"time_to_db_adaptive_job_{target}"] = time_to_db(
                    R.RenderJob(g, W, H, BUDGET, seed=SEED, adaptive=dict(target_levels=target, pass_spp=16, min_spp=64)), gold)
        print(name, json.dumps({k: v for k, v in sc.items() if k != "adaptive"}), flush=True)
        res["scenes"][name] = sc
        g.close()
    if out_path:
        os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
        with open(out_path, "w") as fh:
            json.dump(res, fh, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
