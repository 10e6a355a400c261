#!/usr/bin/env python
"""bench.py — samples/s (and Mrays/s) of the B200 path tracer on the reference's headline scene.

Contract: `python bench.py --gpus N --steps K --warmup W` prints ONE JSON line (rank 0).

Workload (BASELINE.json configs):
  N = 1 : configs[2]  flying_unicorn at 1920x1080, 256 spp (the BVH-heavy scene the target is quoted on).
          The same run also measures every other config as a `configs` block — C1 cornell_box 600x450 64 spp (both
          estimators), C2 cubes 600x450 256 spp MIS off / on, C4 flying_unicorn 3840x2160 4096 spp (one true step),
          C5 progressive cornell_box (frames/s through the streaming job, time to 30 / 35 / 40 dB against the committed
          4096-spp oracle frame) — and `scaling_reference`: the N > 1 frame rendered on this one GPU.
  N > 1 : configs[3]  flying_unicorn at 3840x2160, 256 spp, the SAME frame at every N (strong scaling): 32x32 tiles
          interleaved over the ranks, RGB8 shards all_gathered with NCCL and scattered into scan-line order.  The line
          also carries `weak` (64*N spp: 530.8 M samples per GPU at every N) and, at N = 8, `c4_full`: one true 4096-spp
          step of configs[3].
A "step" is one complete frame: generation -> wavefront iterations until every path has ended -> per-sub-pixel
resolve (clamp, gamma, RGB8).  Nothing is cached between steps (accumulators are cleared, every sample is re-traced,
the seed changes per step).

  value    : whole-job samples/s, scene + BVH resident in HBM, frame left in device memory
  e2e      : the same metric through the host-buffer path, H2D and D2H inside the timed region of every step.
             N = 1: rtb_scene_upload (flattened scene, pinned -> device) + rtb_render into a host frame.
             N > 1: every rank uploads the scene and renders its shard, all_gather over NCCL, rank 0 scatters the shards
             and copies the full frame to pinned host memory; timed by the slowest rank (barrier + synchronize brackets).
  roofline : the kernel with the largest share of the step.  Neither hot kernel is HBM bound: what binds them is
             instruction issue, so `bound` = "issue" (warp-instructions issued per second against 4 schedulers x SMs x
             clock, instruction counts per unit from the committed ncu capture, units and kernel time measured live);
             the HBM view (algorithmic queue bytes) and the FP32 view (SURVEY 8(d) flop model) ride along.
  cpu_baseline / --impl reference : oracle/ (f64 C++ port of the reference, octree traversal, live NEE) on the
             host cores, bounded sample of the same frame.

--dump-outputs DIR (rtb200 arm): after the timed steps, rank 0 writes the RGB8 frame of the last timed step, in scan-line
order, as DIR/frame.npy (float32 [height, width, 3]).  A frame above 64 MB in float32 (the N > 1 frame) is written as a
fixed seeded sample of its pixels instead: DIR/frame_pixels.npy (float64 flat pixel indices y * width + x, ascending) and
DIR/frame_sample.npy (float32 [n, 3]).  The scene and the per-step seeds depend only on the arguments, so two builds run
with the same arguments can be compared output for output (up to the last-level rounding of float atomics).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
SCENES = os.path.join(ROOT, "tests", "golden", "scenes")
SCENE = "flying_unicorn"
METRIC = "samples/sec (Mrays/sec alongside) on flying_unicorn"
UNIT = "samples/s"
# algorithmic HBM bytes of the two hot kernels per unit (DESIGN.md "Kernels and rooflines"):
#   k_shade    per path-queue entry read (camera rays + re-queued paths; a path stays in registers from vertex
#              to vertex while its next hit is analytic): hit 8 + origin/direction/throughput 3 x 16 = 56 B
#              per path-queue entry written: origin/direction/throughput/hit             = 56 B
#              per queued shadow ray written: origin/direction/contribution              = 48 B
#              per NEE contribution added directly: one 16-byte RED                       = 16 B
#   k_traverse per BVH extension ray: origin/direction 32 + hit read 8 + hit write 8     = 48 B
#              per BVH shadow ray   : origin/direction/contribution 48 + one RED 16      = 64 B
#              (+ the LBVH itself, 4 MB, which lives in L1/L2)
SHADE_B_VERTEX, SHADE_B_EXT, SHADE_B_SHQ, SHADE_B_RED = 56.0, 56.0, 48.0, 16.0
TRAV_B_EXT, TRAV_B_SH = 48.0, 64.0
STRONG_FRAME = (3840, 2160, 256)     # the fixed frame of the N > 1 runs
DUMP_BYTES = 64 << 20                # budget of --dump-outputs
DUMP_SAMPLE_PIXELS = 1 << 21         # pixels kept from a frame over budget: 2 Mi x (12 + 8) B = 40 MB


def workload(n_gpus: int):
    if n_gpus == 1:
        return {"width": 1920, "height": 1080, "spp": 256, "name": "flying_unicorn 1920x1080 256spp (configs[2])"}
    w, h, spp = STRONG_FRAME
    return {"width": w, "height": h, "spp": spp,
            "name": f"flying_unicorn {w}x{h} {spp}spp, one frame tile-sharded over {n_gpus} GPUs (configs[3] geometry, fixed frame)"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
            except Exception:
                continue
            for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7), ("sw_power_cap", 8)):
                if len(r) > col and r[col].lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


CPU_BUILD = "oracle/Makefile: g++ -O3 -march=x86-64-v3 -ffp-contract=off (portable across the GPU boxes; not -march=native)"
CPU_SCHED = "dynamic row scheduling over all host threads (the reference's static bands, src/server.rs:166-168, never run in parallel: SURVEY F2)"


def cpu_reference_run(width, height, spp, seconds_target=20.0, threads=None, scene=SCENE, mis=False):
    """Times the oracle port (reference algorithm: octree-faithful traversal, live NEE, f64) on the host
    cores over a bounded sample of the frame: every `stride`-th row at `spp_cpu` spp."""
    from oracle import oracle as O

    threads = threads or os.cpu_count() or 1
    sc = O.OracleScene.from_toml(os.path.join(SCENES, scene + ".toml"))
    sc.set_modes(O.ACCEL_OCTREE_FAITHFUL, O.EST_MIS_DEAD if mis else O.EST_NEE)
    # calibrate on a thin sample, then size the real one for ~seconds_target
    stride = max(1, height // 16)
    t0 = time.perf_counter()
    r = sc.render(width, height, 4, seed=1, nthreads=-threads, row_stride=stride)
    dt = time.perf_counter() - t0
    rate = r["samples"] / max(dt, 1e-6)
    want = rate * seconds_target
    spp_cpu = 16
    rows = max(threads, int(want / (width * spp_cpu)))
    stride = max(1, height // rows)
    t0 = time.perf_counter()
    r = sc.render(width, height, spp_cpu, seed=2, nthreads=-threads, row_stride=stride)
    dt = time.perf_counter() - t0
    n_rows = (height + stride - 1) // stride
    return {"value": r["samples"] / dt, "mrays": r["rays"] / dt / 1e6, "seconds": dt, "cores": threads,
            "sample": f"{n_rows} of {height} rows (every {stride}th) x {width} px at {spp_cpu} spp, "
                      f"{r['samples']} samples, scaled linearly (samples are i.i.d.)"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    wl = workload(args.gpus)
    steps = args.steps
    per_step = max(3.0, min(20.0, 90.0 / (steps + args.warmup)))
    if os.environ.get("RTB_BENCH_CPU_SECONDS"):   # test hook (tests/test_bench_contract.py): a shorter CPU sample
        per_step = float(os.environ["RTB_BENCH_CPU_SECONDS"])
    vals = []
    for _ in range(args.warmup):
        cpu_reference_run(wl["width"], wl["height"], wl["spp"], seconds_target=min(per_step, 3.0))
    t0 = time.perf_counter()
    for _ in range(steps):
        vals.append(cpu_reference_run(wl["width"], wl["height"], wl["spp"], seconds_target=per_step))
    total = time.perf_counter() - t0
    v = sum(x["value"] for x in vals) / len(vals)
    last = vals[-1]
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
        "warmup": args.warmup, "ms_per_step": total / steps * 1e3, "higher_is_better": True,
        "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "reference scene fixtures (tests/golden/scenes), CPU",
        "config": {"workload": wl["name"], "width": wl["width"], "height": wl["height"], "spp": wl["spp"]},
        "mrays_per_s": sum(x["mrays"] for x in vals) / len(vals),
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": last["cores"], "kind": "port", "sample": last["sample"],
                         "build": CPU_BUILD, "scheduling": CPU_SCHED},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    _emit(line)
    return 0


def psnr(a, b):
    import numpy as np

    mse = np.mean((a.astype(np.float64) - b.astype(np.float64)) ** 2)
    return 99.0 if mse == 0 else float(10 * np.log10(255.0 ** 2 / mse))


def dump_frame(out_dir, frame):
    """--dump-outputs: frame (uint8 [h, w, 3], scan-line order) -> out_dir/frame.npy, or a seeded pixel sample when over budget."""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    if frame.size * 4 <= DUMP_BYTES:
        np.save(os.path.join(out_dir, "frame.npy"), frame.astype(np.float32))
        return
    px = frame.reshape(-1, 3)
    idx = np.sort(np.random.default_rng(0).choice(px.shape[0], DUMP_SAMPLE_PIXELS, replace=False))
    np.save(os.path.join(out_dir, "frame_pixels.npy"), idx.astype(np.float64))
    np.save(os.path.join(out_dir, "frame_sample.npy"), px[idx].astype(np.float32))


def measure_configs(R, device, full_c4=True):
    """Every BASELINE.json config that is not the headline frame, on one GPU, in this run."""
    import numpy as np

    out = {}

    def frame_rate(scene, name, w, h, spp, mis, reps):
        scene.render(w, h, min(spp, 16), use_mis=mis)
        best = None
        for i in range(reps):
            t0 = time.perf_counter()
            scene.render(w, h, spp, seed=50 + i, use_mis=mis)
            dt = time.perf_counter() - t0
            st = scene.stats()
            rays = st["rays_primary"] + st["rays_extension"] + st["rays_shadow"]
            r = {"ms": dt * 1e3, "device_ms": st["render_ms"] + st["resolve_ms"], "samples_per_s": st["samples"] / dt,
                 "mrays_per_s": rays / dt / 1e6, "rays_per_sample": rays / max(1, st["samples"]), "iterations": st["iterations"],
                 "timed": "host clock around rtb_render (H2D nothing, D2H frame), best of %d" % reps}
            if best is None or r["ms"] < best["ms"]:
                best = r
        out[name] = best

    cornell = R.Scene.from_toml(os.path.join(SCENES, "cornell_box.toml"), device=device)
    cubes = R.Scene.from_toml(os.path.join(SCENES, "cubes.toml"), device=device)
    frame_rate(cornell, "C1_cornell_box_600x450_64spp_mis_dead_branch", 600, 450, 64, True, 5)
    frame_rate(cornell, "C1_cornell_box_600x450_64spp_nee", 600, 450, 64, False, 5)
    frame_rate(cubes, "C2_cubes_600x450_256spp_mis_off", 600, 450, 256, False, 5)
    frame_rate(cubes, "C2_cubes_600x450_256spp_mis_on_dead_branch", 600, 450, 256, True, 5)
    # C5: progressive cornell_box through the streaming job, 1 sample per pixel per frame (4 frames = reference spp 4)
    gold = None
    try:
        gold = np.load(os.path.join(ROOT, "tests", "golden", "converged", "cornell_box_nee_600x450_4096spp_seed7.npz"))["rgb8"]
    except Exception:
        pass
    W, H, passes = 600, 450, 4096
    for warm in (True, False):
        job = R.RenderJob(cornell, W, H, 64 if warm else passes, seed=3, passes=64 if warm else passes)
        marks, n, nxt = {}, 0, 4
        reached = {30: None, 35: None, 40: None}
        t0 = time.perf_counter()
        for i, f in job.frames():
            n += 1
            if not warm and gold is not None and n >= nxt:      # PSNR on a geometric schedule: it costs more than a frame
                t = time.perf_counter() - t0
                p = psnr(f, gold)
                marks[n] = [round(t * 1e3, 2), round(p, 2)]
                for db in reached:
                    if reached[db] is None and p >= db:
                        reached[db] = {"frames": n, "ms": round(t * 1e3, 2)}
                nxt = max(n + 1, int(n * 1.25))
        dt = time.perf_counter() - t0
        st = job.stats()
        job.close()
    # frames/s without the PSNR bookkeeping in the consumer
    job = R.RenderJob(cornell, W, H, 1024, seed=4, passes=1024)
    t0 = time.perf_counter()
    m = sum(1 for _ in job.frames())
    dt_plain = time.perf_counter() - t0
    job.close()
    out["C5_cornell_box_progressive_600x450"] = {
        "frames_per_s": m / dt_plain, "frames": m, "samples_per_frame": W * H, "first_frame_ms": st["first_record_ms"],
        "api": "rtb_job_begin(passes = spp) + rtb_job_next_frame: every frame resolved on the device and copied to pinned host memory",
        "time_to_psnr_db": reached, "psnr_reference": "tests/golden/converged/cornell_box_nee_600x450_4096spp_seed7.npz (f64 oracle, other seed: its own noise caps the PSNR)",
        "psnr_after_frames_ms_db": marks}
    if full_c4:
        g = R.Scene.from_toml(os.path.join(SCENES, SCENE + ".toml"), device=device)
        frame_rate(g, "C4_flying_unicorn_3840x2160_4096spp_one_gpu", 3840, 2160, 4096, False, 1)
        del g
    return out


_REAL_STDOUT = None


def _stdout_for_json_only():
    """The contract is ONE JSON line on stdout; libraries do not know that (NCCL prints its version line to fd 1 when the box sets
    NCCL_DEBUG=VERSION).  Everything written to fd 1 from here on goes to stderr, the JSON line goes to the saved descriptor."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def _emit(line: dict):
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="rtb200", choices=["rtb200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the configs / scaling_reference / weak / c4_full blocks")
    ap.add_argument("--spp", type=int, default=0, help="override spp (debug only; invalidates the bench line)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the frame of the last timed step to DIR (rtb200 arm)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs needs the rtb200 arm (the reference arm renders a timing-sized row sample)")
    _stdout_for_json_only()
    if args.impl == "reference":
        return run_reference(args)

    import ctypes as C

    import numpy as np
    import torch

    import raytracer_server_b200 as R
    from raytracer_server_b200 import _abi, sharding

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            print(f"bench.py: --gpus {args.gpus} needs torchrun (WORLD_SIZE={world})", file=sys.stderr)
            return 2
    if not torch.cuda.is_available():
        print("bench.py: no CUDA device (there is no CPU fallback for the rtb200 arm)", file=sys.stderr)
        return 2
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=dev)

    wl = workload(world)
    W, H, SPP = wl["width"], wl["height"], args.spp or wl["spp"]
    t_load = time.perf_counter()
    if world > 1:   # the scene and its LBVH are loaded / built on rank 0 and broadcast ONCE (NCCL); the other ranks import the tables
        scene = sharding.broadcast_scene(os.path.join(SCENES, SCENE + ".toml") if rank == 0 else None, device=local_rank, src=0)
        torch.cuda.synchronize(dev)
    else:
        scene = R.Scene.from_toml(os.path.join(SCENES, SCENE + ".toml"), device=local_rank)
    t_load = time.perf_counter() - t_load
    L = _abi.lib()

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(dev)

    class Frame:
        """device buffers of one (w, h) frame geometry on this rank"""

        def __init__(self, w, h):
            self.w, self.h = w, h
            self.stride = sharding.shard_stride(w, h, world)
            self.shard = torch.zeros(self.stride, dtype=torch.uint8, device=dev)
            self.gathered = torch.empty(world * self.stride, dtype=torch.uint8, device=dev) if world > 1 else None
            self.frame = torch.empty((h, w, 3), dtype=torch.uint8, device=dev)
            self.host = torch.empty((h, w, 3), dtype=torch.uint8, pin_memory=True) if rank == 0 else None

    STAT_KEYS = ("samples", "rays_primary", "rays_extension", "rays_shadow", "kernel_launches", "iterations", "rays_bvh", "shadow_bvh", "paths_queued")
    MS_KEYS = ("render_ms", "extend_ms", "shade_ms", "resolve_ms", "bin_ms")

    def step(fr, spp, seed, totals, upload=False, to_host=False):
        """one frame on `world` GPUs: [scene H2D] -> render shard -> [all_gather -> untile on rank 0] -> [frame D2H]"""
        if upload:
            totals["h2d"] = scene.upload()
        p = R.make_params(fr.w, fr.h, spp, seed=seed, rank=rank, world=world)
        scene.render_device(p, fr.shard.data_ptr())
        st = scene.stats()
        for k in STAT_KEYS:
            totals[k] = totals.get(k, 0) + st[k]
        for k in MS_KEYS:
            totals[k] = totals.get(k, 0.0) + st[k]
        src = fr.shard
        if world > 1:
            dist.all_gather_into_tensor(fr.gathered, fr.shard)
            if rank == 0:   # on torch's current stream, right behind the collective: no device-wide synchronisation
                R.host._check(L.rtb_untile_device_async(C.byref(p), C.c_void_p(fr.gathered.data_ptr()), fr.stride, C.c_void_p(fr.frame.data_ptr()),
                                                        local_rank, C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)))
                totals["kernel_launches"] += 1
            src = fr.frame
        if to_host and rank == 0:
            if world > 1:
                fr.host.copy_(src, non_blocking=True)
            else:   # single GPU: the shard IS the frame in tile order; the host-buffer API call (rtb_render) is timed instead
                pass
        if world > 1:
            torch.cuda.synchronize(dev)

    def timed(fr, spp, steps, warmup, seed0, **kw):
        """W untimed + K timed steps, barrier + synchronize on both sides, max over ranks; counters summed over ranks"""
        for i in range(warmup):
            step(fr, spp, seed0 + i, {}, **kw)
        barrier()
        totals = {}
        t0 = time.perf_counter()
        for i in range(steps):
            step(fr, spp, seed0 + warmup + i, totals, **kw)
        barrier()
        elapsed = time.perf_counter() - t0
        job = dict(totals)
        if dist is not None:
            t = torch.tensor([elapsed], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            elapsed = float(t.item())
            c = torch.tensor([float(totals[k]) for k in STAT_KEYS], dtype=torch.float64, device=dev)
            dist.all_reduce(c, op=dist.ReduceOp.SUM)
            job.update(dict(zip(STAT_KEYS, [float(x) for x in c.tolist()])))
            m = torch.tensor([float(totals[k]) for k in MS_KEYS], dtype=torch.float64, device=dev)
            dist.all_reduce(m, op=dist.ReduceOp.MAX)
            job["render_ms_max_rank"] = float(m[0].item())
        return elapsed, job, totals

    def summary(elapsed, job, steps):
        rays = job["rays_primary"] + job["rays_extension"] + job["rays_shadow"]
        return {"samples_per_s": job["samples"] / elapsed, "mrays_per_s": rays / elapsed / 1e6, "ms_per_step": elapsed / max(1, steps) * 1e3,
                "steps": steps}

    # ---------------------------------------------------------------- value: K timed steps of the headline frame
    # The headline frames (path pools of 32 Mi slots) are launched kernel by kernel, with CUDA events around k_traverse / k_shade: that
    # is what the library does for pools above 16 Mi anyway; RTB_NO_GRAPH pins it, so that the per-kernel times the roofline needs are
    # there even under the --spp debug override.  The `configs` block below runs with the library's defaults (graph replay).
    os.environ["RTB_NO_GRAPH"] = "1"
    fr = Frame(W, H)
    clocks = ClockSampler(local_rank)
    for i in range(args.warmup):
        step(fr, SPP, 1000 + i, {})
    barrier()
    if rank == 0:
        clocks.start()
    elapsed, job, totals = timed(fr, SPP, args.steps, 0, 1000 + args.warmup)
    clk = clocks.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:   # before anything else renders into fr
        dump_frame(args.dump_outputs, fr.frame.cpu().numpy() if world > 1 else
                   sharding.untile_numpy(fr.shard.cpu().numpy()[None], W, H, 1))
    value = job["samples"] / elapsed
    rays = job["rays_primary"] + job["rays_extension"] + job["rays_shadow"]

    # ---------------------------------------------------------------- e2e: host buffers, copies inside every step
    e2e_steps = max(1, min(args.steps, 3))
    if world == 1:
        host_frame = np.zeros((H, W, 3), dtype=np.uint8)
        scene.upload()
        scene.render(W, H, SPP, seed=5, out=host_frame)
        t1 = time.perf_counter()
        e2e_samples, h2d = 0, 0
        for i in range(e2e_steps):
            h2d = scene.upload()
            scene.render(W, H, SPP, seed=2000 + i, out=host_frame)
            e2e_samples += scene.stats()["samples"]
        e2e_dt = time.perf_counter() - t1
        d2h = W * H * 3
        e2e_api = "rtb_scene_upload + rtb_render (host RGB8 frame)"
    else:
        e2e_dt, e2e_job, e2e_tot = timed(fr, SPP, e2e_steps, 1, 3000, upload=True, to_host=True)
        e2e_samples, h2d, d2h = e2e_job["samples"], int(e2e_tot.get("h2d", 0)) * world, W * H * 3
        e2e_api = ("every rank: rtb_scene_upload + rtb_render_device (shard); all_gather_into_tensor over NCCL; rank 0: rtb_untile_device_async + "
                   "frame -> pinned host memory; slowest rank")
    e2e_value = e2e_samples / e2e_dt

    extra = {}
    if not args.no_configs and not args.spp:
        if world == 1:
            sw, sh, sspp = STRONG_FRAME
            sfr = Frame(sw, sh)
            el, jb, _ = timed(sfr, sspp, 2, 1, 4000)
            extra["scaling_reference"] = dict(summary(el, jb, 2), workload=f"flying_unicorn {sw}x{sh} {sspp}spp on one GPU: the N > 1 frame, for fixed-frame (strong) scaling")
            del sfr
        else:
            # the N = 1 workload's sample count per GPU (weak scaling, as round 1 reported it)
            el, jb, _ = timed(fr, 64 * world, 2, 1, 5000)
            extra["weak"] = dict(summary(el, jb, 2), workload=f"flying_unicorn {W}x{H} {64 * world}spp: 530.8 M samples per GPU at every N")
            if world == 8:
                el, jb, _ = timed(fr, 4096, 1, 0, 6000)
                extra["c4_full"] = dict(summary(el, jb, 1), workload=f"flying_unicorn {W}x{H} 4096spp (configs[3] in full), one step")

    out = None
    if rank == 0:
        # ---- rooflines of the two hot kernels, measured live over the timed region (CUDA events around every launch,
        # recorded on the render stream inside librtb200 and summed); the one with the larger share is `roofline`
        n_launch = max(1.0, totals["iterations"])
        vertices = totals["rays_primary"] + totals["rays_extension"]      # path vertices shaded == closest-hit rays
        shadow_direct = totals["rays_shadow"] - totals["shadow_bvh"]       # upper bound of the REDs issued by k_shade
        entries_read = totals["rays_primary"] + totals["paths_queued"]     # what k_shade pulls out of the path queue
        shade_bytes = (entries_read * SHADE_B_VERTEX + totals["paths_queued"] * SHADE_B_EXT + totals["shadow_bvh"] * SHADE_B_SHQ
                       + shadow_direct * SHADE_B_RED)
        trav_bytes = totals["rays_bvh"] * TRAV_B_EXT + totals["shadow_bvh"] * TRAV_B_SH
        peaks = {}
        try:
            with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
                peaks = json.load(f)
        except Exception:
            pass
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        prof = {}
        try:
            with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
                prof = json.load(f)
        except Exception:
            pass
        props = torch.cuda.get_device_properties(dev)
        sm_hz = (clk.get("sm_mhz") or 1965.0) * 1e6
        issue_peak = props.multi_processor_count * 4 * sm_hz          # one warp instruction per scheduler and clock
        units = {"k_shade": vertices, "k_traverse": totals["rays_bvh"] + totals["shadow_bvh"]}
        unit_name = {"k_shade": "path vertex", "k_traverse": "LBVH ray (extension + shadow)"}
        per_unit_key = {"k_shade": "k_shade_warp_inst_per_vertex", "k_traverse": "k_traverse_warp_inst_per_bvh_ray"}
        traffic_key = {"k_shade": "k_shade_dram_bytes_per_vertex", "k_traverse": "k_traverse_dram_bytes_per_bvh_ray"}

        def roof(kernel, ms, nbytes):
            secs = ms * 1e-3
            gbs = nbytes / secs / 1e9 if ms > 0 else 0.0
            inst = prof.get(per_unit_key[kernel], 0.0) * units[kernel]          # warp instructions issued in the timed region
            ips = inst / secs if ms > 0 else 0.0
            traffic = prof.get(traffic_key[kernel], 0.0) * units[kernel] / n_launch or None
            return {"kernel": kernel, "bound": "issue", "achieved": ips / 1e9, "peak": issue_peak / 1e9, "unit": "G warp-instructions/s",
                    "frac": ips / issue_peak,
                    "how": f"{prof.get(per_unit_key[kernel])} warp instructions per {unit_name[kernel]} (ncu smsp__inst_executed.sum over one frame / counted units, "
                           f"profiles/traffic.json, build {prof.get('commit')}) x units counted live / kernel time from CUDA events; peak = {props.multi_processor_count} SMs x 4 "
                           f"schedulers x {sm_hz / 1e6:.0f} MHz (median SM clock of this run)",
                    "traffic": traffic, "traffic_source": f"ncu dram__bytes_read.sum + dram__bytes_write.sum per unit on build {prof.get('commit')} (profiles/traffic.json) x this run's units per launch",
                    "issue_active_pct_ncu": prof.get(kernel + "_issue_active_pct"),
                    "lanes_per_instruction_ncu": prof.get(kernel + "_lanes_per_instruction"),
                    "pipe_fma_pct_ncu": prof.get(kernel + "_pipe_fma_pct"), "pipe_alu_pct_ncu": prof.get(kernel + "_pipe_alu_pct"),
                    "hbm": {"bound": "hbm", "achieved": gbs, "peak": hbm_peak, "unit": "GB/s", "frac": gbs / hbm_peak,
                            "algorithmic_bytes_per_launch": nbytes / n_launch,
                            "peak_source": "MEASURED_PEAKS.json" if peaks else "fallback 6650"},
                    "avg_launch_ms": ms / n_launch, "share_of_step": ms / max(totals["render_ms"], 1e-9)}

        roofs = [roof("k_shade", totals["shade_ms"], shade_bytes), roof("k_traverse", totals["extend_ms"], trav_bytes)]
        roofs.sort(key=lambda r: -r["share_of_step"])
        # FP32 view: flop model of SURVEY §8(d) with node visits / triangle tests measured by a counting pass
        pc = R.make_params(640, 360, 16, seed=9, count_work=True)
        cnt_frame = torch.zeros(sharding.shard_stride(640, 360, 1), dtype=torch.uint8, device=dev)
        scene.render_device(pc, cnt_frame.data_ptr())
        cs = scene.stats()
        crays = cs["rays_primary"] + cs["rays_extension"] + cs["rays_shadow"]
        n_node, n_tri = cs["bvh_node_visits"] / crays, cs["bvh_tri_tests"] / crays
        info = scene.info
        flops_per_ray = 14 * info.n_planes + 20 * info.n_spheres + 48 * n_node + 46 * n_tri
        flops_per_vertex = 120.0
        fp32_peak = R.fp32_peak_tflops(local_rank)
        step_s = totals["render_ms"] * 1e-3
        fp32_achieved = ((totals["rays_primary"] + totals["rays_extension"] + totals["rays_shadow"]) * flops_per_ray
                         + vertices * flops_per_vertex) / step_s / 1e12

        cpu = None
        if not args.no_cpu_baseline and world == 1:
            c = cpu_reference_run(W, H, SPP, seconds_target=15.0)
            cpu = {"value": c["value"], "unit": UNIT, "cores": c["cores"], "kind": "port", "sample": c["sample"],
                   "mrays_per_s": c["mrays"], "build": CPU_BUILD, "scheduling": CPU_SCHED}
        os.environ.pop("RTB_NO_GRAPH", None)
        if world == 1 and not args.no_configs and not args.spp:
            extra["configs"] = measure_configs(R, local_rank)

        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": elapsed / max(1, args.steps) * 1e3, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "reference scene fixtures (tests/golden/scenes), Philox seeds per step",
            "config": {"workload": wl["name"], "width": W, "height": H, "spp": SPP},
            "workload_detail": {
                "samples_per_step": W * H * (SPP // 4) * 4,
                "parallelism": f"tiles32x32 interleaved x{world}, one all_gather per frame" if world > 1 else "single GPU",
                "scaling_note": "N > 1 renders ONE fixed frame (3840x2160, 256 spp) at every N; the N = 1 line is configs[2] and carries the fixed frame as scaling_reference",
                "launch_mode": "kernel-by-kernel launches with CUDA events around k_traverse / k_shade (the library's own mode for pools above 16 Mi slots, pinned with RTB_NO_GRAPH=1); the configs block uses the library defaults (CUDA-graph replay for its small frames)", "l2": "no flush needed: every step re-traces the whole frame, streaming ~270 GB through HBM (path / shadow queue entries of the paths that leave registers + the accumulator buffer, cleared per step), far more than the 126 MB L2; only the 4 MB scene + LBVH is meant to stay cache-resident",
                "timing": "host clock between barrier + torch.cuda.synchronize brackets (rtb_render_device returns synchronised), max over ranks; device_ms_per_step = CUDA events on the render stream"},
            "mrays_per_s": rays / elapsed / 1e6,
            "rays_per_sample": rays / max(1.0, job["samples"]),
            "device_ms_per_step": totals["render_ms"] / max(1, args.steps),
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "ms_per_step": e2e_dt / e2e_steps * 1e3, "steps": e2e_steps, "api": e2e_api},
            "gpu_launches": int(job["kernel_launches"]),
            "clocks": clk,
            "roofline": dict(roofs[0], fp32={"achieved": fp32_achieved, "peak": fp32_peak, "unit": "TFLOP/s",
                                             "frac": fp32_achieved / fp32_peak, "flops_per_ray": flops_per_ray,
                                             "flops_per_vertex": flops_per_vertex, "bvh_nodes_per_ray": n_node,
                                             "tri_tests_per_ray": n_tri, "scope": "whole step, flop model of SURVEY 8(d)",
                                             "peak_source": "rtb_fp32_peak FMA chain, this run"}),
            "roofline_other": roofs[1],
            "bvh_ray_fraction": {"extension": totals["rays_bvh"] / max(1.0, vertices),
                                 "shadow": totals["shadow_bvh"] / max(1.0, totals["rays_shadow"])},
            "cpu_baseline": cpu,
            # once per job, outside every timed region.  N = 1: parse TOML + OBJ, flatten, upload, build the LBVH on the device.
            # N > 1: rank 0 does that, exports objects + LBVH tables (rtb_scene_export) and broadcasts the blob over NCCL; the
            # other ranks import it (rtb_scene_import): no parsing, no build, bit-identical tables on every GPU
            "setup": {"scene_load_ms": t_load * 1e3, "lbvh_build_ms": info.build_ms, "lbvh_nodes": info.bvh_nodes, "lbvh_depth": info.bvh_depth,
                      "triangles": info.n_triangles, "broadcast_bytes": int(scene.export().size) if world > 1 else 0,
                      "note": "scene_load_ms includes the first CUDA context use" + ("; rank 0: load + build + export + broadcast" if world > 1 else "")},
        }
        out.update(extra)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0:
        _emit(out)
    return 0


if __name__ == "__main__":
    sys.exit(main())
