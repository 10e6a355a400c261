"""WebSocket host speaking the reference's protocol on top of librtb200 (SURVEY §8(f) rank 1).

Protocol (reference `src/server.rs`):
  * client -> server, text JSON (`ClientMessage`, :121-126):
        {"type": "render", "scene": "<name>", "spp": <int>}      accepted only while the connection is idle (:94-106)
        {"type": "stop_rendering"}                                accepted only while a job runs (:108-111)
    anything else is ignored (:112).  Extension (ignored by the reference's serde structs, so old clients are
    unaffected): "passes": <int> renders progressively and re-sends every record once per pass; "noise": <number> asks
    for adaptive sampling instead — every 32x32 tile stops once its estimated standard error is at most that many 8-bit
    output levels, with "spp" as the budget (rounded down to a multiple of ADAPTIVE_PASS_SPP), and every record is
    re-sent once per pass until all tiles have stopped.
  * server -> client, binary, one message per <= 60 pixels of one screen row (:173-190):
        [0] = 0 (message type)   [1] = n   [2..4] = x u16le   [4..6] = y u16le (row 0 = top)   then n x (r, g, b)
    There is no "done" message; the client counts pixels (test-client/app.tsx:69-70).
  * one job per connection; scenes are shared by all connections (:24); frame size 600 x 450 (:29-30);
    `$PORT`, default 8080 (src/main.rs:16,38); scene names cornell_box, cubes, flying_unicorn (src/main.rs:17).

Differences from the reference, on purpose: malformed JSON (including an "spp" that is not a JSON integer in i32
range, which serde rejects) closes that connection with code 1007 instead of panicking the task (:92); an unknown
scene name is answered with nothing instead of an `unwrap` panic (:100); a request the library refuses (spp beyond the
20-bit sample index) is logged and ignored, the connection stays open.  spp < 4 — negative values included — streams
a black frame exactly like the reference (`num_samples = spp / 4`, :332).

Run:  python -m raytracer_server_b200.server <scenes dir>
"""
from __future__ import annotations

import asyncio
import json
import math
import os
import random
import string
import sys
from typing import Callable, Iterable

SCENE_NAMES = ("cornell_box", "cubes", "flying_unicorn")  # src/main.rs:17
WIDTH, HEIGHT = 600, 450                                   # Server::WIDTH / HEIGHT, src/server.rs:29-30
DEFAULT_PORT = "8080"                                      # src/main.rs:16
ADAPTIVE_PASS_SPP = 16                                     # "noise" requests: samples per pixel per pass ...
ADAPTIVE_MIN_SPP = 64                                      # ... and the least any tile gets (clipped to the budget)


def default_job_factory(scenes: dict, width: int, height: int, accel: int = 0):
    """accel: 0 = LBVH (true nearest hit, the fast path), 1 = the reference's own octrees (ACCEL_OCTREE_REFERENCE: the image the
    Rust binary sends, non-nearest triangles included; 2.4 x slower on flying_unicorn).  `main` reads it from $RTB_ACCEL."""
    from .host import RenderJob

    def make(scene_name: str, spp: int, passes: int = 1, adaptive: dict | None = None):
        scene = scenes.get(scene_name)
        if scene is None:
            return None
        # spp is an i32 in the reference (`ClientMessage::Render`, :123); `num_samples = spp / 4` makes every spp < 4,
        # negative ones included, an empty sample loop: a black frame is streamed (src/server.rs:332-362)
        return RenderJob(scene, width, height, max(0, spp), passes=passes, seed=random.getrandbits(63), accel=accel,
                         adaptive=adaptive)

    return make


class Server:
    def __init__(self, scenes: dict | None = None, *, width: int = WIDTH, height: int = HEIGHT,
                 job_factory: Callable | None = None, log=print):
        self.scenes = scenes or {}
        self.width, self.height = width, height
        self.job_factory = job_factory or default_job_factory(self.scenes, width, height)
        self.connections: set[str] = set()
        self.log = log

    # Server::generate_connection_id, src/server.rs:63-78: five distinct lowercase letters, unique
    def generate_connection_id(self) -> str:
        while True:
            cid = "".join(random.sample(string.ascii_lowercase, 5))
            if cid not in self.connections:
                self.connections.add(cid)
                return cid

    async def handle_connection(self, websocket):
        cid = self.generate_connection_id()
        self.log(f"[{cid}] Accepted connection.")
        state = {"job": None, "task": None}
        try:
            async for msg in websocket:
                if not isinstance(msg, str):
                    continue                                   # only Message::Text is looked at (:90)
                self.log(f"[{cid}] New message: '{msg}'")
                try:
                    req = json.loads(msg)
                    kind = req.get("type") if isinstance(req, dict) else None
                except (ValueError, AttributeError):
                    await websocket.close(code=1007, reason="failed to parse message")
                    break
                running = state["task"] is not None and not state["task"].done()
                if kind == "render" and not running:
                    try:
                        scene_name, spp, passes = req["scene"], req["spp"], req.get("passes", 1)
                        # serde: `scene: String`, `spp: i32` — a JSON string / float / bool / out-of-range number is a parse error
                        if not isinstance(scene_name, str) or type(spp) is not int or not -2 ** 31 <= spp < 2 ** 31 or type(passes) is not int:
                            raise TypeError
                        passes = max(1, passes)
                        adaptive = self._adaptive_options(req["noise"], spp) if "noise" in req else None
                    except (KeyError, TypeError, ValueError, OverflowError):
                        await websocket.close(code=1007, reason="failed to parse message")
                        break
                    try:
                        if adaptive is not None:
                            budget, opts = adaptive
                            job = self.job_factory(scene_name, budget, 1, adaptive=opts)
                        else:
                            job = self.job_factory(scene_name, spp, passes)
                    except RuntimeError as e:                  # the library refused the request (RtbError): not a reason to drop the client
                        self.log(f"[{cid}] render request refused: {e}")
                        continue
                    if job is None:
                        self.log(f"[{cid}] unknown scene '{scene_name}'")
                        continue
                    state["job"] = job
                    self.log(f"[{cid}] Rendering...")
                    state["task"] = asyncio.create_task(self._run_job(cid, websocket, job))
                elif kind == "stop_rendering" and running:
                    state["job"].stop()
                    self.log(f"[{cid}] Render cancelled.")
        finally:
            if state["job"] is not None:
                state["job"].stop()                            # closed socket cancels the job (:212-216)
            if state["task"] is not None:
                try:
                    await state["task"]
                except Exception:
                    pass
            self.connections.discard(cid)
            self.log(f"[{cid}] Disconnected.")

    @staticmethod
    def _adaptive_options(noise, spp: int) -> tuple[int, dict] | None:
        """(budget, adaptive options) of the job a "noise" request asks for, or None when the budget is too small for two
        passes (a plain job then renders the frame).  Raises ValueError unless noise is a finite non-negative JSON number."""
        if type(noise) not in (int, float) or not math.isfinite(noise) or noise < 0:
            raise ValueError("noise")
        budget = max(0, spp) // ADAPTIVE_PASS_SPP * ADAPTIVE_PASS_SPP
        if budget < 2 * ADAPTIVE_PASS_SPP:
            return None
        return budget, {"target_levels": float(noise), "pass_spp": ADAPTIVE_PASS_SPP, "min_spp": min(ADAPTIVE_MIN_SPP, budget)}

    async def _run_job(self, cid: str, websocket, job):
        """RenderJob::run: forward the job's records as binary messages; the GPU call runs in a worker thread."""
        loop = asyncio.get_running_loop()
        it = iter(job.messages())
        sentinel = object()

        def next_batch(n=128):
            out = []
            for _ in range(n):
                m = next(it, sentinel)
                if m is sentinel:
                    return out, True
                out.append(m)
            return out, False

        try:
            done = False
            while not done:
                batch, done = await loop.run_in_executor(None, next_batch)
                for m in batch:
                    await websocket.send(m)
        except Exception:
            job.stop()                                         # AlreadyClosed / ConnectionClosed -> cancel (:212-216)
        finally:
            cancelled_early = await loop.run_in_executor(None, job.close)
            if not cancelled_early:
                self.log(f"[{cid}] Done rendering.")

    async def listen(self, port: int | str, host: str = "0.0.0.0", ready: asyncio.Future | None = None):
        import websockets

        async with websockets.serve(self.handle_connection, host, int(port), max_size=1 << 20) as srv:
            self.log(f"Listening on port {port}.")
            if ready is not None and not ready.done():
                ready.set_result(srv)
            await asyncio.Future()


def load_scenes(scenes_dir: str, device: int = 0) -> dict:
    """src/main.rs:30-36: the three hard-coded scenes from <dir>/<name>.toml, meshes from <dir>/assets."""
    from .host import LoadTomlError, Scene

    scenes = {}
    for name in SCENE_NAMES:
        try:
            scenes[name] = Scene.from_toml(os.path.join(scenes_dir, name + ".toml"), os.path.join(scenes_dir, "assets"), device)
        except LoadTomlError as e:                            # src/main.rs:45-54: message + exit(1)
            print(f"failed to load scene {name}: {e}", file=sys.stderr)
            sys.exit(1)
    return scenes


def main(argv=None):
    argv = sys.argv[1:] if argv is None else argv
    if len(argv) != 1:
        print("usage: python -m raytracer_server_b200.server <scenes dir>", file=sys.stderr)
        return 2
    scenes = load_scenes(argv[0])
    port = os.environ.get("PORT", DEFAULT_PORT)
    accel = 1 if os.environ.get("RTB_ACCEL", "lbvh").lower() in ("octree", "reference", "1") else 0
    asyncio.run(Server(scenes, job_factory=default_job_factory(scenes, WIDTH, HEIGHT, accel)).listen(port))
    return 0


if __name__ == "__main__":
    sys.exit(main())
