"""Host-side objects over the C ABI: Context (one GPU), Scene (uploaded world + BVH), render calls.

Mirrors what the reference's worker() does per job (ray-tracer-slave/src/main.rs:32-106):
`Scene` = `req.world` + `BVH::build`, `render_division` = the rayon row loop, its return value =
`ImageSlice.image`.  Every call goes through librt_b200.so; errors raise RtError (the reference
`.unwrap()`s instead).
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _abi
from ._abi import INTERSECT_AUTO, INTERSECT_BRUTE, INTERSECT_BVH, RtParams, RtStats  # noqa: F401
from .scenes import SPHERE_DTYPE, TRIANGLE_DTYPE


class RtError(RuntimeError):
    def __init__(self, status: int, message: str):
        super().__init__(f"{_abi.STATUS_NAMES.get(status, status)}: {message}")
        self.status = status
        self.message = message


def make_params(width, height, divisions=1, division_no=0, spp=0, max_bounces=0, seed=0,
                cam_origin=(0.0, 0.0, 0.0), aperture=0.0, focus_distance=0.0, field_of_view=0.0,
                focal_length=0.0, intersector=INTERSECT_AUTO, collect_counters=False, explicit=()) -> RtParams:
    """Zero fields mean the reference's literals (spp 100, max_bounces 10, aperture 0.1, ...), except the fields named
    in `explicit` ("max_bounces": 0 = camera rays only; "aperture": 0 = pinhole), whose zero is taken as given."""
    p = RtParams()
    p.flags = ((_abi.PARAM_MAX_BOUNCES_EXPLICIT if "max_bounces" in explicit else 0)
               | (_abi.PARAM_APERTURE_EXPLICIT if "aperture" in explicit else 0))
    p.width, p.height, p.divisions, p.division_no = width, height, divisions, division_no
    p.spp, p.max_bounces, p.seed = spp, max_bounces, seed
    p.cam_origin[:] = [float(c) for c in cam_origin]
    p.aperture, p.focus_distance, p.field_of_view, p.focal_length = aperture, focus_distance, field_of_view, focal_length
    p.intersector = intersector
    p.collect_counters = 1 if collect_counters else 0
    return p


def _ptr(a):
    return None if a is None or a.size == 0 else a.ctypes.data_as(C.c_void_p)


def bvh_build_host(spheres=None, triangles=None, world_index=None):
    """Host-only BVH build (no GPU): (rank per world position, node count, depth)."""
    L = _abi.lib()
    sp = np.ascontiguousarray(spheres if spheres is not None else np.zeros(0, SPHERE_DTYPE), dtype=SPHERE_DTYPE)
    tr = np.ascontiguousarray(triangles if triangles is not None else np.zeros(0, TRIANGLE_DTYPE), dtype=TRIANGLE_DTYPE)
    wi = None if world_index is None else np.ascontiguousarray(world_index, dtype=np.uint32)
    rank = np.zeros(len(sp) + len(tr), dtype=np.uint32)
    nn, d = C.c_uint32(), C.c_uint32()
    rc = L.rt_bvh_build_host(_ptr(sp), len(sp), _ptr(tr), len(tr), _ptr(wi), _ptr(rank), C.byref(nn), C.byref(d))
    if rc != 0:
        raise RtError(rc, L.rt_last_error(None).decode())
    return rank, nn.value, d.value


class Context:
    """One GPU, one stream; single owner (same contract as the reference's single worker thread)."""

    def __init__(self, device: int = 0):
        self._lib = _abi.lib()
        h = C.c_void_p()
        rc = self._lib.rt_init(device, C.byref(h))
        if rc != 0:
            raise RtError(rc, self._lib.rt_last_error(None).decode())
        self._h = h
        self.device = device

    # -- plumbing -------------------------------------------------------------------------------
    def _check(self, rc):
        if rc != 0:
            raise RtError(rc, self._lib.rt_last_error(self._h).decode())

    def close(self):
        if getattr(self, "_h", None):
            for p in getattr(self, "_pinned", []):
                self._lib.rt_host_free(self._h, p)
            self._pinned = []
            self._lib.rt_shutdown(self._h)
            self._h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def device_info(self):
        sm, clk, smem = C.c_int(), C.c_int(), C.c_int()
        name = C.create_string_buffer(64)
        self._check(self._lib.rt_device_info(self._h, C.byref(sm), C.byref(clk), C.byref(smem), name))
        return {"sm_count": sm.value, "clock_khz": clk.value, "smem_optin": smem.value, "name": name.value.decode()}

    def measure_fp32_peak(self):
        tf, ms = C.c_double(), C.c_float()
        self._check(self._lib.rt_measure_fp32_peak(self._h, C.byref(tf), C.byref(ms)))
        return tf.value, ms.value

    def l2_flush(self, nbytes: int, timed: bool = False):
        """Queue a write of `nbytes` (> L2) in front of the next render on this context's stream; timed → its ms."""
        ms = C.c_float()
        self._check(self._lib.rt_l2_flush(self._h, nbytes, C.byref(ms) if timed else None))
        return ms.value if timed else None

    def sync(self):
        self._check(self._lib.rt_sync(self._h))

    @property
    def stream(self) -> int:
        return int(self._lib.rt_stream(self._h) or 0)

    # -- scene ----------------------------------------------------------------------------------
    def scene(self, spheres=None, triangles=None, world_index=None) -> "Scene":
        return Scene(self, spheres, triangles, world_index)

    # -- pinned host buffers ----------------------------------------------------------------------
    def pinned_empty(self, shape) -> np.ndarray:
        """uint8 array in page-locked host memory (full-rate D2H target)."""
        n = int(np.prod(shape))
        p = C.c_void_p()
        self._check(self._lib.rt_host_alloc(self._h, n, C.byref(p)))
        buf = (C.c_uint8 * n).from_address(p.value)
        arr = np.frombuffer(buf, dtype=np.uint8).reshape(shape)
        self._pinned = getattr(self, "_pinned", [])
        self._pinned.append(p)
        return arr

    # -- render -----------------------------------------------------------------------------------
    @staticmethod
    def _out_buffer(out, shape):
        """A caller-supplied destination must be exactly the bytes the library will write."""
        if out is None:
            return np.empty(shape, dtype=np.uint8)
        if not isinstance(out, np.ndarray) or out.dtype != np.uint8 or not out.flags["C_CONTIGUOUS"] or not out.flags["WRITEABLE"]:
            raise RtError(_abi.RT_ERR_INVALID_ARG, "out must be a writable C-contiguous uint8 numpy array")
        return out

    def render_division(self, scene: "Scene", params: RtParams, out: np.ndarray | None = None, want_stats=False):
        """Band `params.division_no` → uint8 (height/divisions, width, 3); row 0 = top of the band."""
        div = params.divisions or 1
        if params.height % div != 0:
            raise RtError(_abi.RT_ERR_INVALID_ARG, f"height {params.height} is not a multiple of divisions {div}")
        rows = params.height // div
        out = self._out_buffer(out, (rows, params.width, 3))
        st = RtStats()
        self._check(self._lib.rt_render_division(self._h, scene._h, C.byref(params), out.ctypes.data_as(C.c_void_p),
                                                 out.nbytes, C.byref(st)))
        return (out, st.as_dict()) if want_stats else out

    def render_divisions(self, scene: "Scene", params: RtParams, division_nos, out: np.ndarray | None = None,
                         want_stats=False):
        """Bands `division_nos` of one job in one launch → uint8 (n, height/divisions, width, 3); out[k] is
        render_division of band division_nos[k] (params.division_no is ignored)."""
        div = params.divisions or 1
        if params.height % div != 0:
            raise RtError(_abi.RT_ERR_INVALID_ARG, f"height {params.height} is not a multiple of divisions {div}")
        nos = np.asarray(division_nos, dtype=np.int64).reshape(-1)
        if ((nos < 0) | (nos > 0xFFFFFFFF)).any():
            raise RtError(_abi.RT_ERR_INVALID_ARG, "division numbers must fit 32 bits unsigned")
        nos = np.ascontiguousarray(nos, dtype=np.uint32)
        out = self._out_buffer(out, (len(nos), params.height // div, params.width, 3))
        st = RtStats()
        self._check(self._lib.rt_render_divisions(self._h, scene._h, C.byref(params), _ptr(nos), len(nos),
                                                  out.ctypes.data_as(C.c_void_p), out.nbytes, C.byref(st)))
        return (out, st.as_dict()) if want_stats else out

    def render_divisions_json(self, scene: "Scene", params: RtParams, division_nos, id: str, want_stats=False):
        """Bands `division_nos` of one job as the ImageSlice bodies the slave POSTs to /result, written on the device
        (rt_render_divisions_json): body k is wire.ImageSlice(division_nos[k], band, id).to_json().encode() of the band
        render_divisions gives; the RGB never reaches the host."""
        div = params.divisions or 1
        if params.height % div != 0:
            raise RtError(_abi.RT_ERR_INVALID_ARG, f"height {params.height} is not a multiple of divisions {div}")
        nos = np.asarray(division_nos, dtype=np.int64).reshape(-1)
        if ((nos < 0) | (nos > 0xFFFFFFFF)).any():
            raise RtError(_abi.RT_ERR_INVALID_ARG, "division numbers must fit 32 bits unsigned")
        nos = np.ascontiguousarray(nos, dtype=np.uint32)
        buf = np.empty(max(1, len(nos) * self._lib.rt_slice_json_bound(params.height // div, params.width)), np.uint8)
        lens = np.zeros(max(1, len(nos)), dtype=np.uintp)
        st = RtStats()
        self._check(self._lib.rt_render_divisions_json(self._h, scene._h, C.byref(params), _ptr(nos), len(nos),
                                                       str(id).encode(), _ptr(buf), buf.nbytes,
                                                       lens.ctypes.data_as(C.POINTER(C.c_size_t)), C.byref(st)))
        ends = np.cumsum(lens[: len(nos)])
        bodies = [buf[e - n: e].tobytes() for e, n in zip(ends.tolist(), lens[: len(nos)].tolist())]
        return (bodies, st.as_dict()) if want_stats else bodies

    def parse_world_json(self, text, start: int = 0):
        """The "world" array at text[start:] (bytes or str; leading JSON whitespace allowed) parsed on the device
        (rt_world_parse_json): (wire.World, offset in text just past the array's ']'), the arrays
        wire.parse_render_info builds.  None when the text is outside the device grammar; the host parser then decides."""
        from .wire import World

        data = text.encode("utf-8", "surrogatepass") if isinstance(text, str) else bytes(text)
        if not 0 <= start <= len(data):
            raise RtError(_abi.RT_ERR_INVALID_ARG, f"start {start} outside the text")
        n_bytes = len(data) - start
        base = C.c_void_p(C.cast(C.c_char_p(data), C.c_void_p).value + start)
        cap = self._lib.rt_world_json_max_objects(n_bytes)
        sp, tr = np.empty(cap, SPHERE_DTYPE), np.empty(cap, TRIANGLE_DTYPE)
        wi = np.empty(cap, np.uint32)
        ns, nt, used = C.c_uint32(), C.c_uint32(), C.c_size_t()
        rc = self._lib.rt_world_parse_json(self._h, base, n_bytes, _ptr(sp), _ptr(tr), _ptr(wi), cap, C.byref(ns),
                                           C.byref(nt), C.byref(used))
        if rc == _abi.RT_ERR_UNSUPPORTED:
            return None
        self._check(rc)
        n = ns.value + nt.value
        return World(sp[: ns.value].copy(), tr[: nt.value].copy(), wi[:n].copy()), start + used.value

    def parse_obj(self, body: bytes, obj_size: int):
        """The controller's /upload body (OBJ = body[:obj_size], MTL = the rest) built into its world on the device
        (rt_obj_build_world): the TRIANGLE_DTYPE array obj.build_world returns, byte for byte.  None when the body is
        outside the device grammar, which includes every body the host rejects; obj.build_world then decides."""
        data = body if isinstance(body, bytes) else bytes(body)
        if not 0 <= obj_size <= len(data):
            raise RtError(_abi.RT_ERR_INVALID_ARG, f"obj_size {obj_size} outside the body")
        cap = self._lib.rt_obj_max_triangles(obj_size)
        tr = np.empty(max(cap, 1), TRIANGLE_DTYPE)
        n = C.c_uint32()
        rc = self._lib.rt_obj_build_world(self._h, C.cast(C.c_char_p(data), C.c_void_p), len(data), obj_size,
                                          tr.ctypes.data_as(C.c_void_p), cap, C.byref(n))
        if rc == _abi.RT_ERR_UNSUPPORTED:
            return None
        self._check(rc)
        return tr[: n.value].copy()

    def render_frame(self, scene: "Scene", params: RtParams, out: np.ndarray | None = None, want_stats=False):
        """All divisions in one launch → uint8 (height, width, 3)."""
        out = self._out_buffer(out, (params.height, params.width, 3))
        st = RtStats()
        self._check(self._lib.rt_render_frame(self._h, scene._h, C.byref(params), out.ctypes.data_as(C.c_void_p),
                                              out.nbytes, C.byref(st)))
        return (out, st.as_dict()) if want_stats else out

    def encode_jpeg(self, frame: np.ndarray, quality: int = 90, want_ms=False):
        """Baseline JPEG of a uint8 (height, width, 3) frame, encoded on this context's GPU (rt_jpeg_encode): the bytes
        PIL's save(format="JPEG", quality=quality) writes.  want_ms: also the device time of the encode."""
        frame = np.ascontiguousarray(frame, dtype=np.uint8)
        if frame.ndim != 3 or frame.shape[2] != 3:
            raise RtError(_abi.RT_ERR_INVALID_ARG, f"frame must be (height, width, 3), not {frame.shape}")
        h, w = frame.shape[:2]
        buf = np.empty(self._lib.rt_jpeg_bound(w, h), dtype=np.uint8)
        n, ms = C.c_size_t(0), C.c_float(0.0)
        self._check(self._lib.rt_jpeg_encode(self._h, _ptr(frame), w, h, int(quality), _ptr(buf), buf.nbytes,
                                             C.byref(n), C.byref(ms)))
        data = buf[: n.value].tobytes()
        return (data, ms.value) if want_ms else data

    def render_frame_jpeg(self, scene: "Scene", params: RtParams, quality: int = 90, want_stats=False):
        """render_frame, then the frame encoded as JPEG on the device (rt_render_frame_jpeg): the bytes of
        encode_jpeg(render_frame(...)); the RGB frame never reaches the host."""
        return render_frame_jpeg([self], [scene], params, quality=quality, want_stats=want_stats)

    def render_tiles_device(self, scene: "Scene", params: RtParams, tile_rank: int, tile_ranks: int, frame_dev: int,
                            sync=True, want_stats=False):
        """This rank's tiles of the whole frame into a device (possibly peer-mapped) frame buffer."""
        st = RtStats()
        self._check(self._lib.rt_render_tiles_device(self._h, scene._h, C.byref(params), tile_rank, tile_ranks,
                                                     C.c_void_p(frame_dev), 1 if sync else 0, C.byref(st)))
        return st.as_dict() if want_stats else None

    def render_tiles_collect(self, scene: "Scene", params: RtParams, tile_rank: int, tile_ranks: int, frame_dev: int,
                             seq: int, out: np.ndarray | None, want_stats=False):
        """Frame owner: this rank's tiles into its frame, and the whole frame (all ranks' slabs, as they complete) into
        `out` while they render."""
        if out is not None:
            out = self._out_buffer(out, None)
        st = RtStats()
        self._check(self._lib.rt_render_tiles_collect(self._h, scene._h, C.byref(params), tile_rank, tile_ranks,
                                                      C.c_void_p(frame_dev), int(seq),
                                                      None if out is None else out.ctypes.data_as(C.c_void_p),
                                                      0 if out is None else out.nbytes, C.byref(st)))
        return st.as_dict() if want_stats else None

    # -- progressive rendering ---------------------------------------------------------------------------
    def accum(self, params: RtParams) -> "Accum":
        """Sample state (device memory, 96 bytes per pixel) of the band `params` selects, every pixel at sample 0."""
        return Accum(self, params)

    def render_samples(self, scene: "Scene", acc: "Accum", n: int, out: np.ndarray | None = None, download=True,
                       want_stats=False):
        """Advance every pixel of `acc` by `n` samples of its chain.  The band as it now stands (byte-identical to
        render_division at spp = acc.samples) goes to `out` (None: a new array); download=False skips the copy and
        returns None in its place."""
        if download:
            out = self._out_buffer(out, (acc.rows, acc.width, 3))
        else:
            out = None
        st = RtStats()
        self._check(self._lib.rt_render_samples(self._h, scene._h, acc._h, int(n),
                                                None if out is None else out.ctypes.data_as(C.c_void_p),
                                                0 if out is None else out.nbytes, C.byref(st)))
        return (out, st.as_dict()) if want_stats else out

    def render_progressive(self, scene: "Scene", params: RtParams, schedule=(1, 1, 2, 4, 8)):
        """Preview that improves: yields (samples_done, frame) after each chunk of `schedule` samples; each frame equals
        render_division at spp = samples_done."""
        with self.accum(params) as acc:
            for n in schedule:
                frame = self.render_samples(scene, acc, n)
                yield acc.samples, frame

    # -- shared frame (one NVLink box, one process per GPU) ----------------------------------------------
    def frame_alloc(self, nbytes: int):
        p = C.c_void_p()
        handle = (C.c_uint8 * 64)()
        self._check(self._lib.rt_frame_alloc(self._h, nbytes, C.byref(p), handle))
        return p.value, bytes(handle)

    def frame_open(self, handle: bytes) -> int:
        p = C.c_void_p()
        hb = (C.c_uint8 * 64).from_buffer_copy(handle)
        self._check(self._lib.rt_frame_open(self._h, hb, C.byref(p)))
        return p.value

    def frame_close(self, dev: int):
        self._check(self._lib.rt_frame_close(self._h, C.c_void_p(dev)))

    def frame_free(self, dev: int):
        self._check(self._lib.rt_frame_free(self._h, C.c_void_p(dev)))

    def frame_download(self, dev: int, out: np.ndarray):
        out = self._out_buffer(out, None)
        self._check(self._lib.rt_frame_download(self._h, C.c_void_p(dev), out.ctypes.data_as(C.c_void_p), out.nbytes))
        return out

    def frame_wait_consumed(self, dev: int, nbytes: int, seq: int):
        """Non-owner rank: later work on this context's stream waits until the owner has collected frame `seq`."""
        self._check(self._lib.rt_frame_wait_consumed(self._h, C.c_void_p(dev), nbytes, int(seq)))

    def frame_collect(self, dev: int, params: RtParams, seq: int, out: np.ndarray | None = None):
        """Frame owner: wait (on the device) until frame number `seq` of the buffer is complete — every rank's kernel
        counts the pixels it finishes in the frame's control block — and stream finished slabs into `out` meanwhile."""
        if out is not None:
            out = self._out_buffer(out, None)
        self._check(self._lib.rt_frame_collect(self._h, C.c_void_p(dev), C.byref(params), int(seq),
                                               None if out is None else out.ctypes.data_as(C.c_void_p),
                                               0 if out is None else out.nbytes))
        return out


def render_frame_multi(ctxs, scenes, params: RtParams, out: np.ndarray | None = None, want_stats=False):
    """One frame on several GPUs from this process (rt_render_frame_multi): context i renders rank i's tiles of its own
    copy of the scene straight into context 0's frame over peer access; finished slabs stream to `out`."""
    if len(ctxs) != len(scenes) or not ctxs:
        raise RtError(_abi.RT_ERR_INVALID_ARG, "one scene per context")
    out = Context._out_buffer(out, (params.height, params.width, 3))
    n = len(ctxs)
    ch = (C.c_void_p * n)(*[c._h for c in ctxs])
    sh = (C.c_void_p * n)(*[s._h for s in scenes])
    st = RtStats()
    ctxs[0]._check(ctxs[0]._lib.rt_render_frame_multi(ch, sh, n, C.byref(params), out.ctypes.data_as(C.c_void_p),
                                                      out.nbytes, C.byref(st)))
    return (out, st.as_dict()) if want_stats else out


def render_frame_jpeg(ctxs, scenes, params: RtParams, quality: int = 90, want_stats=False):
    """The frame of render_frame (one context) or render_frame_multi (several) as JPEG bytes, encoded on ctxs[0]'s GPU
    where the frame lies (rt_render_frame_jpeg).  Stats: the render's, total_ms including the encode."""
    if len(ctxs) != len(scenes) or not ctxs:
        raise RtError(_abi.RT_ERR_INVALID_ARG, "one scene per context")
    L = ctxs[0]._lib
    n = len(ctxs)
    ch = (C.c_void_p * n)(*[c._h for c in ctxs])
    sh = (C.c_void_p * n)(*[s._h for s in scenes])
    buf = np.empty(L.rt_jpeg_bound(params.width, params.height), dtype=np.uint8)
    size, st = C.c_size_t(0), RtStats()
    ctxs[0]._check(L.rt_render_frame_jpeg(ch, sh, n, C.byref(params), int(quality), _ptr(buf), buf.nbytes, C.byref(size),
                                          C.byref(st)))
    data = buf[: size.value].tobytes()
    return (data, st.as_dict()) if want_stats else data


def render_samples_multi(ctxs, scenes, accs, n: int, out: np.ndarray | None = None, download=True, want_stats=False):
    """One progressive frame on several contexts (rt_render_samples_multi): accs[i] (a whole-frame Accum of ctxs[i])
    holds the chains of rank i's tiles; every pixel advances by `n` samples and the frame as it now stands (byte-identical
    to render_frame at spp = accs[0].samples) goes to `out` (None: a new array); download=False skips the copy and returns
    None in its place."""
    if not ctxs or not (len(ctxs) == len(scenes) == len(accs)):
        raise RtError(_abi.RT_ERR_INVALID_ARG, "one scene and one accum per context")
    k = len(ctxs)
    out = Context._out_buffer(out, (accs[0].rows, accs[0].width, 3)) if download else None
    ch = (C.c_void_p * k)(*[c._h for c in ctxs])
    sh = (C.c_void_p * k)(*[s._h for s in scenes])
    ah = (C.c_void_p * k)(*[a._h for a in accs])
    st = RtStats()
    ctxs[0]._check(ctxs[0]._lib.rt_render_samples_multi(ch, sh, ah, k, int(n),
                                                        None if out is None else out.ctypes.data_as(C.c_void_p),
                                                        0 if out is None else out.nbytes, C.byref(st)))
    return (out, st.as_dict()) if want_stats else out


class Accum:
    """Resumable per-pixel sample chains of one frame or division (rt_accum): chunks rendered with
    Context.render_samples add up to the frame render_division renders at the cumulative sample count."""

    def __init__(self, ctx: Context, params: RtParams):
        self._ctx = ctx
        self._h = None
        div = params.divisions or 1
        if params.height % div != 0:
            raise RtError(_abi.RT_ERR_INVALID_ARG, f"height {params.height} is not a multiple of divisions {div}")
        h = C.c_void_p()
        ctx._check(ctx._lib.rt_accum_create(ctx._h, C.byref(params), C.byref(h)))
        self._h = h
        self.width, self.rows = params.width, params.height // div

    @property
    def samples(self) -> int:
        n = C.c_uint32()
        self._ctx._check(self._ctx._lib.rt_accum_samples(self._h, C.byref(n)))
        return n.value

    def reset(self, params: RtParams | None = None):
        """Back to sample 0, optionally with new params of the same size and band (a camera move, another seed)."""
        self._ctx._check(self._ctx._lib.rt_accum_reset(self._ctx._h, self._h, None if params is None else C.byref(params)))

    def read_linear(self) -> np.ndarray:
        """float32 (rows, width, 3): sum / samples per channel, before the gamma and 8-bit quantisation."""
        out = np.empty((self.rows, self.width, 3), dtype=np.float32)
        self._ctx._check(self._ctx._lib.rt_accum_read_linear(self._ctx._h, self._h, out.ctypes.data_as(C.c_void_p),
                                                             out.nbytes))
        return out

    def close(self):
        if self._h and self._ctx._h:
            self._ctx._lib.rt_accum_destroy(self._ctx._h, self._h)
        self._h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Scene:
    """Device-resident world: primitive SoA + BVH (replaces req.world + BVH::build, main.rs:60-61)."""

    def __init__(self, ctx: Context, spheres=None, triangles=None, world_index=None):
        self._ctx = ctx
        self._h = None
        sp = np.ascontiguousarray(spheres if spheres is not None else np.zeros(0, SPHERE_DTYPE), dtype=SPHERE_DTYPE)
        tr = np.ascontiguousarray(triangles if triangles is not None else np.zeros(0, TRIANGLE_DTYPE), dtype=TRIANGLE_DTYPE)
        wi = None if world_index is None else np.ascontiguousarray(world_index, dtype=np.uint32)
        if wi is not None and len(wi) != len(sp) + len(tr):
            raise RtError(_abi.RT_ERR_INVALID_ARG, "world_index length must be n_spheres + n_triangles")
        h = C.c_void_p()
        ctx._check(ctx._lib.rt_scene_create(ctx._h, _ptr(sp), len(sp), _ptr(tr), len(tr), _ptr(wi), C.byref(h)))
        self._h = h
        self.n_spheres, self.n_triangles = len(sp), len(tr)

    def update(self, spheres=None, triangles=None) -> "Scene":
        """Replace the world with one of the same shape (as many spheres and triangles as created; the creation's
        world_index still applies): geometry, materials and emission may all change.  Later renders are byte-identical
        to those of a scene created from the new world; an Accum with samples of the old one needs reset()."""
        sp = np.ascontiguousarray(spheres if spheres is not None else np.zeros(0, SPHERE_DTYPE), dtype=SPHERE_DTYPE)
        tr = np.ascontiguousarray(triangles if triangles is not None else np.zeros(0, TRIANGLE_DTYPE), dtype=TRIANGLE_DTYPE)
        if (len(sp), len(tr)) != (self.n_spheres, self.n_triangles):
            raise RtError(_abi.RT_ERR_INVALID_ARG, f"{len(sp)} spheres and {len(tr)} triangles for a scene of "
                                                   f"{self.n_spheres} and {self.n_triangles}")
        self._ctx._check(self._ctx._lib.rt_scene_update(self._ctx._h, self._h, _ptr(sp), len(sp), _ptr(tr), len(tr)))
        return self

    def info(self):
        n, nn, d = C.c_uint32(), C.c_uint32(), C.c_uint32()
        rank = np.zeros(self.n_spheres + self.n_triangles, dtype=np.uint32)
        self._ctx._check(self._ctx._lib.rt_scene_info(self._h, C.byref(n), C.byref(nn), C.byref(d), _ptr(rank)))
        return {"n_prims": n.value, "n_nodes": nn.value, "depth": d.value, "rank": rank}

    def wait_ready(self):
        """Block until the tie-break tables (reference-topology tree, built beside the upload) are on the device."""
        self._ctx._check(self._ctx._lib.rt_scene_wait_ready(self._ctx._h, self._h))
        return self

    @property
    def device_bytes(self) -> int:
        return int(self._ctx._lib.rt_scene_device_bytes(self._h))

    def close(self):
        if self._h and self._ctx._h:
            self._ctx._lib.rt_scene_destroy(self._ctx._h, self._h)
        self._h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
