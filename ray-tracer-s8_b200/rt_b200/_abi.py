"""ctypes binding of include/rt_b200.h (librt_b200.so).

The library is the product; this module only declares its entry points.  It fails loudly when the
shared object is missing — there is no Python / CPU fallback for any render call.
"""
from __future__ import annotations

import ctypes as C
import os

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
LIB_DIR = os.path.normpath(os.path.join(PKG_DIR, "..", "lib"))
# RT_B200_LIB=exp selects the experiments build (product + the A/B kernels of csrc/experiments/, `make exp`): tooling and
# the variant-agreement test only.  The product library is the default and carries no A/B code.
_sel = os.environ.get("RT_B200_LIB", "")
LIB_PATH = (_sel if "/" in _sel else           # a development build under another name (A/B measurements)
            os.path.join(LIB_DIR, "librt_b200_exp.so" if _sel == "exp" else "librt_b200.so"))

RT_OK = 0
RT_ERR_INVALID_ARG = -1
RT_ERR_EMPTY_SCENE = -2
RT_ERR_NO_DEVICE = -3
RT_ERR_CUDA = -4
RT_ERR_BVH = -5
RT_ERR_UNSUPPORTED = -6
RT_ERR_NOMEM = -7
RT_ERR_INTERNAL = -8
RT_ERR_TIMEOUT = -9
STATUS_NAMES = {
    0: "RT_OK", -1: "RT_ERR_INVALID_ARG", -2: "RT_ERR_EMPTY_SCENE", -3: "RT_ERR_NO_DEVICE", -4: "RT_ERR_CUDA",
    -5: "RT_ERR_BVH", -6: "RT_ERR_UNSUPPORTED", -7: "RT_ERR_NOMEM", -8: "RT_ERR_INTERNAL", -9: "RT_ERR_TIMEOUT",
}
PARAM_MAX_BOUNCES_EXPLICIT, PARAM_APERTURE_EXPLICIT = 1, 2

INTERSECT_AUTO, INTERSECT_BRUTE, INTERSECT_BVH = 0, 1, 2


class RtParams(C.Structure):
    _fields_ = [
        ("width", C.c_uint32), ("height", C.c_uint32), ("divisions", C.c_uint32), ("division_no", C.c_uint32),
        ("spp", C.c_uint32), ("max_bounces", C.c_uint32), ("seed", C.c_uint64),
        ("cam_origin", C.c_float * 3),
        ("aperture", C.c_float), ("focus_distance", C.c_float), ("field_of_view", C.c_float),
        ("focal_length", C.c_float),
        ("intersector", C.c_uint32), ("collect_counters", C.c_uint32), ("flags", C.c_uint32),
    ]


class RtStats(C.Structure):
    _fields_ = [
        ("rays", C.c_uint64), ("primary", C.c_uint64), ("slab_tests", C.c_uint64), ("sphere_tests", C.c_uint64),
        ("sphere_exact", C.c_uint64), ("sphere_hits", C.c_uint64), ("tri_tests", C.c_uint64),
        ("tri_stage", C.c_uint64 * 3), ("tri_hits", C.c_uint64), ("shades_sphere", C.c_uint64),
        ("shades_tri", C.c_uint64), ("emissive", C.c_uint64), ("sky", C.c_uint64),
        ("active_lane_iters", C.c_uint64), ("total_lane_iters", C.c_uint64),
        ("kernel_ms", C.c_float), ("total_ms", C.c_float),
        ("intersector_used", C.c_uint32), ("kernel_launches", C.c_uint32),
        ("grid_ctas", C.c_uint32), ("cta_threads", C.c_uint32), ("ctas_per_sm", C.c_uint32),
        ("scene_in_smem", C.c_uint32), ("dyn_smem_bytes", C.c_uint32), ("redo_pixels", C.c_uint32),
    ]

    def as_dict(self):
        d = {}
        for name, _ in self._fields_:
            v = getattr(self, name)
            d[name] = list(v) if hasattr(v, "__len__") else v
        return d


# every symbol include/rt_b200.h declares (tests check that the library exports all of them)
EXPORTS = [
    "rt_abi_version", "rt_init", "rt_shutdown", "rt_last_error", "rt_scene_create", "rt_scene_destroy",
    "rt_scene_info", "rt_render_division", "rt_render_frame", "rt_render_tiles_device", "rt_sync", "rt_stream",
    "rt_host_alloc", "rt_host_free", "rt_frame_alloc", "rt_frame_open", "rt_frame_close", "rt_frame_free",
    "rt_frame_download", "rt_measure_fp32_peak", "rt_device_info", "rt_bvh_build_host", "rt_struct_sizes", "rt_scene_device_bytes",
    "rt_scene_wait_ready", "rt_render_frame_multi", "rt_frame_collect", "rt_render_tiles_collect", "rt_frame_wait_consumed", "rt_l2_flush",
    "rt_accum_create", "rt_accum_destroy", "rt_accum_reset", "rt_accum_samples", "rt_render_samples", "rt_accum_read_linear",
]
# only in the experiments build (csrc/experiments/rt_experiments_api.h)
EXPERIMENT_EXPORTS = ["rt_debug_trace_bench"]

_lib = None


class LibraryMissing(RuntimeError):
    pass


def lib():
    """Load librt_b200.so; raise LibraryMissing (never fall back) when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise LibraryMissing(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(make -C ray-tracer-s8_b200/csrc). There is no CPU fallback."
        )
    L = C.CDLL(LIB_PATH)
    vp, u32, i32, sz = C.c_void_p, C.c_uint32, C.c_int, C.c_size_t
    pp = C.POINTER(C.c_void_p)
    L.rt_abi_version.restype = i32
    L.rt_init.argtypes = [i32, pp]
    L.rt_init.restype = i32
    L.rt_shutdown.argtypes = [vp]
    L.rt_shutdown.restype = None
    L.rt_last_error.argtypes = [vp]
    L.rt_last_error.restype = C.c_char_p
    L.rt_scene_create.argtypes = [vp, vp, u32, vp, u32, vp, pp]
    L.rt_scene_create.restype = i32
    L.rt_scene_destroy.argtypes = [vp, vp]
    L.rt_scene_destroy.restype = None
    L.rt_scene_info.argtypes = [vp, C.POINTER(u32), C.POINTER(u32), C.POINTER(u32), vp]
    L.rt_scene_info.restype = i32
    L.rt_render_division.argtypes = [vp, vp, C.POINTER(RtParams), vp, sz, C.POINTER(RtStats)]
    L.rt_render_division.restype = i32
    L.rt_render_frame.argtypes = [vp, vp, C.POINTER(RtParams), vp, sz, C.POINTER(RtStats)]
    L.rt_render_frame.restype = i32
    L.rt_render_tiles_device.argtypes = [vp, vp, C.POINTER(RtParams), u32, u32, vp, i32, C.POINTER(RtStats)]
    L.rt_render_tiles_device.restype = i32
    L.rt_sync.argtypes = [vp]
    L.rt_sync.restype = i32
    L.rt_stream.argtypes = [vp]
    L.rt_stream.restype = vp
    L.rt_host_alloc.argtypes = [vp, sz, pp]
    L.rt_host_alloc.restype = i32
    L.rt_host_free.argtypes = [vp, vp]
    L.rt_host_free.restype = None
    L.rt_frame_alloc.argtypes = [vp, sz, pp, vp]
    L.rt_frame_alloc.restype = i32
    L.rt_frame_open.argtypes = [vp, vp, pp]
    L.rt_frame_open.restype = i32
    L.rt_frame_close.argtypes = [vp, vp]
    L.rt_frame_close.restype = i32
    L.rt_frame_free.argtypes = [vp, vp]
    L.rt_frame_free.restype = i32
    L.rt_frame_download.argtypes = [vp, vp, vp, sz]
    L.rt_frame_download.restype = i32
    L.rt_measure_fp32_peak.argtypes = [vp, C.POINTER(C.c_double), C.POINTER(C.c_float)]
    L.rt_measure_fp32_peak.restype = i32
    if hasattr(L, "rt_debug_trace_bench"):
        L.rt_debug_trace_bench.argtypes = [vp, vp, C.c_void_p, C.c_uint64, i32, C.POINTER(C.c_uint64), C.POINTER(C.c_float),
                                           C.POINTER(C.c_float), C.POINTER(C.c_uint64)]
        L.rt_debug_trace_bench.restype = i32
    L.rt_scene_wait_ready.argtypes = [vp, vp]
    L.rt_scene_wait_ready.restype = i32
    L.rt_render_frame_multi.argtypes = [pp, pp, u32, C.POINTER(RtParams), vp, sz, C.POINTER(RtStats)]
    L.rt_render_frame_multi.restype = i32
    L.rt_render_tiles_collect.argtypes = [vp, vp, C.POINTER(RtParams), u32, u32, vp, C.c_uint64, vp, sz, C.POINTER(RtStats)]
    L.rt_render_tiles_collect.restype = i32
    L.rt_l2_flush.argtypes = [vp, sz, C.POINTER(C.c_float)]
    L.rt_l2_flush.restype = i32
    L.rt_frame_wait_consumed.argtypes = [vp, vp, sz, C.c_uint64]
    L.rt_frame_wait_consumed.restype = i32
    L.rt_frame_collect.argtypes = [vp, vp, C.POINTER(RtParams), C.c_uint64, vp, sz]
    L.rt_frame_collect.restype = i32
    L.rt_device_info.argtypes = [vp, C.POINTER(i32), C.POINTER(i32), C.POINTER(i32), C.c_char_p]
    L.rt_device_info.restype = i32
    L.rt_bvh_build_host.argtypes = [vp, u32, vp, u32, vp, vp, C.POINTER(u32), C.POINTER(u32)]
    L.rt_bvh_build_host.restype = i32
    L.rt_scene_device_bytes.argtypes = [vp]
    L.rt_scene_device_bytes.restype = sz
    L.rt_accum_create.argtypes = [vp, C.POINTER(RtParams), pp]
    L.rt_accum_create.restype = i32
    L.rt_accum_destroy.argtypes = [vp, vp]
    L.rt_accum_destroy.restype = None
    L.rt_accum_reset.argtypes = [vp, vp, C.POINTER(RtParams)]
    L.rt_accum_reset.restype = i32
    L.rt_accum_samples.argtypes = [vp, C.POINTER(u32)]
    L.rt_accum_samples.restype = i32
    L.rt_render_samples.argtypes = [vp, vp, vp, u32, vp, sz, C.POINTER(RtStats)]
    L.rt_render_samples.restype = i32
    L.rt_accum_read_linear.argtypes = [vp, vp, vp, sz]
    L.rt_accum_read_linear.restype = i32
    L.rt_struct_sizes.argtypes = [C.POINTER(sz)]
    L.rt_struct_sizes.restype = None
    sizes = (sz * 4)()
    L.rt_struct_sizes(sizes)
    if list(sizes) != [36, 56, C.sizeof(RtParams), C.sizeof(RtStats)]:
        raise RuntimeError(f"struct layout mismatch between librt_b200.so {list(sizes)} and this binding")
    _lib = L
    return L
