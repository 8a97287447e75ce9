"""Controller: mirror of ray-tracer-controller/src/main.rs on top of the GPU slave.

  POST /upload/{obj_size}/   body = OBJ bytes ++ MTL bytes → job id (uuid4 text)      (main.rs:22-77)
  POST /result               body = ImageSlice JSON        → "slice saved. thank you slave."   (main.rs:79-93)
  POST /poll                 body = job id                 → JPEG(90) | status text   (main.rs:95-142)

Same literals as the reference: 1920x1080, 20 divisions (main.rs:33-36), the same status strings.  Dispatch is one of
  * the reference's: HTTP `RenderInfo` POSTs to `http://slave:8081`, results arrive on /result (main.rs:47-75);
  * `worker=`: the divisions of a job are rendered in-process by one `rt_b200.slave.Worker` (one GPU, scene uploaded once);
  * `devices=[...]`: the tile scheduler — the whole frame in ONE call over all listed GPUs (`rt_render_frame_multi`:
    every GPU renders an interleaved share of the 8x4 tiles straight into GPU 0's frame over NVLink), then cut into
    the job's divisions so /poll stitches them exactly as it stitches slave slices (main.rs:109-119).
/poll's JPEG(90) is encoded on the GPU where there is one: in `devices=` mode the frame is encoded where it was rendered
(`rt_render_frame_jpeg`) and never reaches the host as RGB; in `worker=` mode the stitched frame is encoded with the
worker's context (`rt_jpeg_encode`).  The bytes are the same as PIL's, which the HTTP-slave mode keeps using.
/upload builds the world on the GPU in the same two modes (`Context.parse_obj`: the first GPU's context, or the worker's),
falling back to obj.build_world's host code when the device declines; the HTTP-slave mode parses on the host.
GPU work from concurrent /upload requests is serialised (one rt_ctx has one owner at a time).
"""
from __future__ import annotations

import io
import threading
import urllib.request
import uuid
from http.server import BaseHTTPRequestHandler, ThreadingHTTPServer

import numpy as np

from . import obj as objmod
from . import wire

WIDTH, HEIGHT, DIVISIONS = 1920, 1080, 20          # main.rs:33-36
SLAVE_URL = "http://slave:8081"                    # main.rs:56
SAVED_TEXT = "slice saved. thank you slave."       # main.rs:92


class Controller:
    def __init__(self, worker=None, slave_url: str = SLAVE_URL, width=WIDTH, height=HEIGHT, divisions=DIVISIONS,
                 devices=None, spp: int = 0, max_bounces: int = 0, seed: int = 0):
        self.worker, self.slave_url = worker, slave_url
        self.width, self.height, self.divisions = width, height, divisions
        self.jobs: dict = {}          # id → {"meta": RenderMeta, "result": {division_no: uint8 array}}
        self.lock = threading.Lock()
        self.gpu_lock = threading.Lock()   # the multi-GPU renderer's contexts: one frame at a time
        self.multi = None
        self.spp, self.max_bounces, self.seed = spp, max_bounces, seed
        if devices is not None:
            from . import multi

            self.multi = multi.MultiDeviceRenderer(list(devices))

    def close(self):
        if self.multi is not None:
            self.multi.close()
            self.multi = None

    def _render_all_gpus(self, triangles, meta: "wire.RenderMeta"):
        """devices= mode: one frame over all GPUs, returned as the job's division slices."""
        from . import api

        p = api.make_params(meta.width, meta.height, spp=self.spp, max_bounces=self.max_bounces, seed=self.seed)
        with self.gpu_lock:
            scenes = self.multi.scenes(None, triangles, np.arange(len(triangles), dtype=np.uint32))
            try:
                frame = self.multi.render(scenes, p)
            finally:
                for sc in scenes:
                    sc.close()
        rows = meta.height // meta.divisions          # main.rs:55-56
        return [wire.ImageSlice(d, frame[d * rows:(d + 1) * rows].reshape(-1), meta.id) for d in range(meta.divisions)]

    def _render_all_gpus_jpeg(self, triangles, meta: "wire.RenderMeta") -> bytes:
        """devices= mode: one frame over all GPUs, encoded as JPEG(90) on the first GPU, where the frame lies."""
        from . import api

        p = api.make_params(meta.width, meta.height, spp=self.spp, max_bounces=self.max_bounces, seed=self.seed)
        with self.gpu_lock:
            scenes = self.multi.scenes(None, triangles, np.arange(len(triangles), dtype=np.uint32))
            try:
                return self.multi.render_jpeg(scenes, p, quality=90)
            finally:
                for sc in scenes:
                    sc.close()

    def _obj_parser(self):
        """The device OBJ parser of this mode (None: host only), taken under the lock of the context it uses."""
        if self.multi is not None:
            ctx, lock = self.multi.ctxs[0], self.gpu_lock
        else:
            ctx, lock = getattr(self.worker, "ctx", None), getattr(self.worker, "lock", None)
        if getattr(ctx, "parse_obj", None) is None or lock is None:
            return None

        def parse(data, obj_size):
            with lock:
                return ctx.parse_obj(data, obj_size)
        return parse

    # -- /upload ---------------------------------------------------------------------------------------
    def upload(self, body: bytes, obj_size: int) -> str:
        job_id = str(uuid.uuid4())
        meta = wire.RenderMeta(self.height, self.width, self.divisions, job_id)
        with self.lock:
            self.jobs[job_id] = {"meta": meta, "result": {}}
        triangles = objmod.build_world(body, obj_size, parser=self._obj_parser())   # obj::build_world (main.rs:46)
        if self.multi is not None:
            if self.height % self.divisions != 0:
                raise ValueError(f"height {self.height} is not a multiple of divisions {self.divisions}")
            jpeg = self._render_all_gpus_jpeg(triangles, meta)
            with self.lock:
                if job_id in self.jobs:
                    self.jobs[job_id]["jpeg"] = jpeg
        elif self.worker is not None:
            world = wire.World(np.zeros(0, wire.SPHERE_DTYPE), triangles, np.arange(len(triangles), dtype=np.uint32))
            infos = [wire.RenderInfo(world, meta, d) for d in range(self.divisions)]
            # all divisions in one call (rt_render_divisions) when the worker can; any object with render() still works
            render_many = getattr(self.worker, "render_many", None)
            for sl in render_many(infos) if render_many else map(self.worker.render, infos):
                self.result(sl)
        else:
            for d in range(self.divisions):                      # join_all over 0..divisions (main.rs:47-75)
                text = wire.render_info_to_json(None, triangles, meta, d)
                req = urllib.request.Request(self.slave_url, data=text.encode(),
                                             headers={"Content-Type": "application/json"}, method="POST")
                urllib.request.urlopen(req, timeout=600).read()
        return job_id

    # -- /result ---------------------------------------------------------------------------------------
    def result(self, sl: wire.ImageSlice) -> str:
        with self.lock:
            job = self.jobs.get(sl.id)
            if job is not None:
                job["result"][sl.division_no] = np.asarray(sl.image, dtype=np.uint8).reshape(-1)
        return SAVED_TEXT

    # -- /poll -------------------------------------------------------------------------------------------
    def poll(self, text: str):
        """→ (bytes, is_image)."""
        try:
            job_id = str(uuid.UUID(text.strip()))
        except ValueError:
            return b"Invalid Uuid", False
        with self.lock:
            job = self.jobs.get(job_id)
            if job is None:
                return b"No such job", False
            if "jpeg" in job:                        # devices= mode: the whole frame, already encoded
                del self.jobs[job_id]
                return job["jpeg"], True
            have = sum(1 for d in range(job["meta"].divisions) if d in job["result"])
            if have < job["meta"].divisions:
                return f"Job not finished yet {have}/{job['meta'].divisions}".encode(), False
            frame = np.concatenate([job["result"][d] for d in range(job["meta"].divisions)])   # sorted by division_no
            del self.jobs[job_id]                                                                # main.rs:122
        frame = frame.reshape(job["meta"].height, job["meta"].width, 3)
        ctx = getattr(self.worker, "ctx", None)
        if ctx is not None:                          # worker= mode: encoded on the worker's GPU, same bytes as PIL
            with self.worker.lock:
                return ctx.encode_jpeg(frame, 90), True
        return encode_jpeg(frame, 90), True


def encode_jpeg(frame: np.ndarray, quality: int = 90) -> bytes:
    """Host encoder of the HTTP-slave mode (no GPU context here): libjpeg's defaults, the bytes rt_jpeg_encode writes."""
    from PIL import Image  # image 0.24's JPEG encoder in the reference; any baseline JPEG encoder here

    buf = io.BytesIO()
    Image.fromarray(frame, "RGB").save(buf, format="JPEG", quality=quality)
    return buf.getvalue()


def serve(controller: Controller, host="0.0.0.0", port=8080, ready: threading.Event | None = None,
          stop: threading.Event | None = None):
    class Handler(BaseHTTPRequestHandler):
        def _send(self, data: bytes, ctype="text/plain; charset=utf-8", code=200):
            self.send_response(code)
            self.send_header("Content-Type", ctype)
            self.send_header("Content-Length", str(len(data)))
            self.end_headers()
            self.wfile.write(data)

        def do_POST(self):  # noqa: N802
            body = self.rfile.read(int(self.headers.get("Content-Length") or 0))
            parts = [p for p in self.path.split("/") if p]
            try:
                if len(parts) == 2 and parts[0] == "upload":
                    self._send(controller.upload(body, int(parts[1])).encode())
                elif parts == ["result"]:
                    self._send(controller.result(wire.ImageSlice.from_json(body)).encode())
                elif parts == ["poll"]:
                    data, is_img = controller.poll(body.decode(errors="replace"))
                    self._send(data, "image/jpeg" if is_img else "text/plain; charset=utf-8")
                else:
                    self.send_error(404)
            except (objmod.ObjError, wire.WireError, ValueError) as e:
                self.send_error(400, str(e))

        def log_message(self, *a):
            pass

    srv = ThreadingHTTPServer((host, port), Handler)
    if ready is not None:
        ready.port = srv.server_address[1]
        ready.set()
    if stop is not None:
        threading.Thread(target=lambda: (stop.wait(), srv.shutdown()), daemon=True).start()
    try:
        srv.serve_forever()
    finally:
        srv.server_close()
    return srv
