"""GPU slave: the reference slave's worker() and HTTP shell on top of the C ABI.

Mirrors ray-tracer-slave/src/main.rs:
  * `Worker.render(RenderInfo) -> ImageSlice`  = the body of worker() (main.rs:37-90): camera + BVH +
    render of band `division_no`, bytes in `ImageSlice.image`.  The scene upload + BVH build is cached by
    `render_meta.id`, so the `divisions` requests of one job share one upload (the reference rebuilds its
    BVH per request, main.rs:60).
  * `serve()` = main() + index() (main.rs:148-174): `POST /` with a RenderInfo body answers
    "i'll get you a slice at once" immediately and queues the job for the single worker thread, which
    POSTs the ImageSlice JSON to `http://master:8080/result` (main.rs:85-101).  The worker thread takes every request
    already queued with the one it waited for and renders those of one job together (`Worker.render_many_json`, one
    `rt_render_divisions_json` call, which also writes the ImageSlice bodies on the GPU); each still gets its own
    ImageSlice POST.  The request's world is parsed on the worker's GPU when it is in serde's layout (`Worker.parse`).
spp / max_bounces / camera default to the reference's literals (main.rs:39-51).
"""
from __future__ import annotations

import queue
import threading
import urllib.request
import zlib
from collections import OrderedDict
from http.server import BaseHTTPRequestHandler, ThreadingHTTPServer

import numpy as np

from . import api, wire

ACK_TEXT = "i'll get you a slice at once"      # main.rs:153
MASTER_RESULT_URL = "http://master:8080/result"  # main.rs:94
JSON_LIMIT = 500_000_000                          # main.rs:167


class Worker:
    """One GPU context; jobs are rendered strictly one at a time (main.rs:34-35)."""

    def __init__(self, device: int = 0, spp: int = 0, max_bounces: int = 0, seed: int = 0, cache_size: int = 4,
                 intersector: int = api.INTERSECT_AUTO):
        self.ctx = api.Context(device)
        self.spp, self.max_bounces, self.seed, self.intersector = spp, max_bounces, seed, intersector
        self._scenes: "OrderedDict[tuple, api.Scene]" = OrderedDict()
        self._cache_size = cache_size
        self.scene_uploads = 0
        # one rt_ctx = one owner at a time (include/rt_b200.h): callers on several threads (the controller's in-process
        # mode under a threading HTTP server) are serialised here
        self.lock = threading.Lock()

    @staticmethod
    def _world_key(info: wire.RenderInfo):
        """Job id + a checksum of the world: every RenderInfo carries its own world (lib.rs:25-30), so a client that
        reuses an id with other geometry must not get the cached scene."""
        w = info.world
        crc = 0
        for a in (w.spheres, w.triangles, w.world_index):
            if a is not None and len(a):
                crc = zlib.crc32(np.ascontiguousarray(a).view(np.uint8).reshape(-1), crc)
        return (info.render_meta.id, 0 if w.spheres is None else len(w.spheres),
                0 if w.triangles is None else len(w.triangles), crc)

    def _scene_for(self, info: wire.RenderInfo) -> api.Scene:
        key = self._world_key(info)
        sc = self._scenes.get(key)
        if sc is None:
            w = info.world
            sc = self.ctx.scene(w.spheres, w.triangles, w.world_index)
            self.scene_uploads += 1
            self._scenes[key] = sc
            while len(self._scenes) > self._cache_size:
                _, old = self._scenes.popitem(last=False)
                old.close()
        else:
            self._scenes.move_to_end(key)
        return sc

    def render(self, info: wire.RenderInfo, want_stats: bool = False):
        m = info.render_meta
        p = api.make_params(m.width, m.height, divisions=m.divisions, division_no=info.division_no, spp=self.spp,
                            max_bounces=self.max_bounces, seed=self.seed, intersector=self.intersector)
        with self.lock:
            out = self.ctx.render_division(self._scene_for(info), p, want_stats=want_stats)
        img, st = out if want_stats else (out, None)
        sl = wire.ImageSlice(info.division_no, np.ascontiguousarray(img).reshape(-1), m.id)
        return (sl, st) if want_stats else sl

    def render_many(self, infos, want_stats: bool = False):
        """Requests of one world and one (width, height, divisions) in one call (rt_render_divisions): one ImageSlice per
        request, in order, each equal to render(info)'s.  A division requested twice is rendered once.  The world is
        infos[0]'s (the caller groups by _world_key, which checksums it)."""
        m = infos[0].render_meta
        key = (m.id, m.width, m.height, m.divisions)
        if any((i.render_meta.id, i.render_meta.width, i.render_meta.height, i.render_meta.divisions) != key for i in infos):
            raise ValueError("render_many takes requests of one job: one id, width, height and divisions")
        nos = list(dict.fromkeys(i.division_no for i in infos))
        p = api.make_params(m.width, m.height, divisions=m.divisions, spp=self.spp, max_bounces=self.max_bounces,
                            seed=self.seed, intersector=self.intersector)
        with self.lock:
            out = self.ctx.render_divisions(self._scene_for(infos[0]), p, nos, want_stats=want_stats)
        imgs, st = out if want_stats else (out, None)
        at = {d: k for k, d in enumerate(nos)}
        slices = [wire.ImageSlice(i.division_no, imgs[at[i.division_no]].reshape(-1), i.render_meta.id) for i in infos]
        return (slices, st) if want_stats else slices

    def render_many_json(self, infos):
        """render_many, as the ImageSlice bodies the slave POSTs (bytes, one per request, in order), written on the device
        by rt_render_divisions_json: each equals render(info).to_json().encode()."""
        to_json = getattr(self.ctx, "render_divisions_json", None)
        if to_json is None:  # a context without the device writer (a stand-in): the host encoder, same bytes
            return [sl.to_json().encode() for sl in self.render_many(infos)]
        m = infos[0].render_meta
        key = (m.id, m.width, m.height, m.divisions)
        if any((i.render_meta.id, i.render_meta.width, i.render_meta.height, i.render_meta.divisions) != key for i in infos):
            raise ValueError("render_many_json takes requests of one job: one id, width, height and divisions")
        nos = list(dict.fromkeys(i.division_no for i in infos))
        p = api.make_params(m.width, m.height, divisions=m.divisions, spp=self.spp, max_bounces=self.max_bounces,
                            seed=self.seed, intersector=self.intersector)
        with self.lock:
            bodies = to_json(self._scene_for(infos[0]), p, nos, m.id)
        at = {d: k for k, d in enumerate(nos)}
        return [bodies[at[i.division_no]] for i in infos]

    def parse(self, body: str | bytes) -> wire.RenderInfo:
        """wire.parse_render_info with the world parsed on this worker's GPU when the device grammar covers it (same
        result, same WireError)."""
        parse_world = getattr(self.ctx, "parse_world_json", None)
        if parse_world is None:  # a context without the device parser (a stand-in)
            return wire.parse_render_info(body)

        def world_parser(data, start):
            with self.lock:
                return parse_world(data, start)

        return wire.parse_render_info(body, world_parser=world_parser)

    def render_json(self, body: str | bytes) -> str:
        """RenderInfo JSON in → ImageSlice JSON out."""
        return self.render(wire.parse_render_info(body)).to_json()

    def close(self):
        for sc in self._scenes.values():
            sc.close()
        self._scenes.clear()
        self.ctx.close()


def _post(url: str, body: str | bytes, timeout: float = 60.0) -> str:
    data = body if isinstance(body, bytes) else body.encode()
    req = urllib.request.Request(url, data=data, headers={"Content-Type": "application/json"}, method="POST")
    with urllib.request.urlopen(req, timeout=timeout) as r:
        return r.read().decode(errors="replace")


def serve(host: str = "0.0.0.0", port: int = 8081, result_url: str = MASTER_RESULT_URL, worker: Worker | None = None,
          post=_post, ready: threading.Event | None = None, stop: threading.Event | None = None):
    """Run the slave endpoint until `stop` is set (or forever).  Returns the server object after shutdown."""
    wk = worker or Worker()
    jobs: "queue.Queue[wire.RenderInfo | None]" = queue.Queue()  # crossbeam unbounded channel (main.rs:159)

    def post_body(body):
        try:
            post(result_url, body)
        except Exception as e:  # the reference unwrap()s and dies; we log and keep serving
            print(f"[rt_b200.slave] job failed: {e}", flush=True)

    def render_alone(info):
        try:
            sl = wk.render(info)
        except Exception as e:
            print(f"[rt_b200.slave] job failed: {e}", flush=True)
            return
        post_body(sl.to_json())

    def worker_loop():
        while True:
            info = jobs.get()
            if info is None:
                return
            # every request already queued goes along: the controller POSTs a job's divisions at once, and one launch
            # over several bands keeps the GPU busier than one launch per band
            batch, stopping = [info], False
            while True:
                try:
                    nxt = jobs.get_nowait()
                except queue.Empty:
                    break
                if nxt is None:
                    stopping = True
                    break
                batch.append(nxt)
            groups: dict = {}  # insertion order: groups in the arrival order of their first request
            for i in batch:
                m = i.render_meta
                groups.setdefault((Worker._world_key(i), m.width, m.height, m.divisions), []).append(i)
            for g in groups.values():
                try:
                    bodies = wk.render_many_json(g)
                except Exception as e:
                    if len(g) == 1:
                        print(f"[rt_b200.slave] job failed: {e}", flush=True)
                    else:  # a request that fails on its own (a bad division_no) must not sink the others
                        for i in g:
                            render_alone(i)
                    continue
                for body in bodies:
                    post_body(body)
            if stopping:
                return

    class Handler(BaseHTTPRequestHandler):
        def do_POST(self):  # noqa: N802
            if self.path != "/":
                self.send_error(404)
                return
            n = int(self.headers.get("Content-Length") or 0)
            if n > JSON_LIMIT:
                self.send_error(413)
                return
            try:
                info = wk.parse(self.rfile.read(n))
            except wire.WireError as e:
                self.send_error(400, str(e))
                return
            jobs.put(info)
            data = ACK_TEXT.encode()
            self.send_response(200)
            self.send_header("Content-Type", "text/plain; charset=utf-8")
            self.send_header("Content-Length", str(len(data)))
            self.end_headers()
            self.wfile.write(data)

        def log_message(self, *a):
            pass

    srv = ThreadingHTTPServer((host, port), Handler)
    t = threading.Thread(target=worker_loop, daemon=True)
    t.start()
    if ready is not None:
        ready.port = srv.server_address[1]
        ready.set()
    if stop is not None:
        threading.Thread(target=lambda: (stop.wait(), srv.shutdown()), daemon=True).start()
    try:
        srv.serve_forever()
    finally:
        jobs.put(None)
        t.join(timeout=30)
        srv.server_close()
        if worker is None:
            wk.close()
    return srv


if __name__ == "__main__":
    serve()
