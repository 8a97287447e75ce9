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

    def trace_bench(self, scene: "Scene", params: RtParams, max_rays: int, with_big: bool = True, sort: bool = False):
        """Development aid (experiments build, RT_B200_LIB=exp): the nearest-hit query alone over the recorded queries of
        one frame (csrc/experiments/rt_trace_bench.cuh)."""
        if not hasattr(self._lib, "rt_debug_trace_bench"):
            raise RtError(_abi.RT_ERR_UNSUPPORTED, "rt_debug_trace_bench exists only in librt_b200_exp.so (RT_B200_LIB=exp)")
        n, bad = C.c_uint64(), C.c_uint64()
        ms_ww, ms_sm = C.c_float(), C.c_float()
        self._check(self._lib.rt_debug_trace_bench(self._h, scene._h, C.byref(params), int(max_rays), (1 if with_big else 0) + (2 if sort else 0),
                                                   C.byref(n), C.byref(ms_ww), C.byref(ms_sm), C.byref(bad)))
        return {"rays": n.value, "ms_while_while": ms_ww.value, "ms_state_machine": ms_sm.value, "mismatches": bad.value}

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

    def render_frame(self, scene: "Scene", params: RtParams, out: np.ndarray | None = None, want_stats=False):
        """All divisions in one launch → uint8 (height, width, 3)."""
        out = self._out_buffer(out, (params.height, params.width, 3))
        st = RtStats()
        self._check(self._lib.rt_render_frame(self._h, scene._h, C.byref(params), out.ctypes.data_as(C.c_void_p),
                                              out.nbytes, C.byref(st)))
        return (out, st.as_dict()) if want_stats else out

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
