"""rt_b200 — host side of the B200-native render path for ray-tracer-s8's slave.

`api`    : Context / Scene / render calls over the C ABI (include/rt_b200.h, librt_b200.so)
`scenes` : deterministic synthetic scenes (BASELINE.json configs)
`wire`   : the reference's JSON wire types (RenderInfo / RenderMeta / ImageSlice)
`slave`  : mirror of the reference slave's worker() and HTTP shell on top of the GPU path
`multi`  : tile scheduler over the GPUs of one box (torch.distributed plumbing)
`obj`    : OBJ + MTL ingest as the controller does it (ray-tracer-controller/src/obj.rs)
`controller` : mirror of the controller's /upload, /result, /poll on top of the GPU slave
"""
from . import scenes  # noqa: F401
from .api import (  # noqa: F401
    INTERSECT_AUTO, INTERSECT_BRUTE, INTERSECT_BVH, Accum, Context, RtError, RtParams, RtStats, Scene, make_params,
    render_frame_multi,
)
