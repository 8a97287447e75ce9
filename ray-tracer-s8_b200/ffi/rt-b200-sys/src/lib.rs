//! FFI binding + safe wrapper of `include/rt_b200.h`.
//!
//! The slave's `worker()` (ray-tracer-slave/src/main.rs:32-106) keeps its request/response shell and calls
//! [`Context::scene`] once per job and [`Context::render_division`] in place of the rayon loop
//! (main.rs:53-83).  See INTEGRATION.md for the patch.
#![allow(non_camel_case_types)]

use std::ffi::CStr;
use std::os::raw::{c_char, c_int, c_void};
use std::ptr;

#[repr(C)]
pub struct rt_ctx {
    _private: [u8; 0],
}
#[repr(C)]
pub struct rt_accum {
    _private: [u8; 0],
}
#[repr(C)]
pub struct rt_scene {
    _private: [u8; 0],
}

/// `Sphere {radius, center, p_albedo_at, p_roughness_at, p_emission_at}` (shapes/sphere.rs:13-20)
#[repr(C)]
#[derive(Clone, Copy, Debug, Default)]
pub struct rt_sphere {
    pub center: [f32; 3],
    pub radius: f32,
    pub albedo: [f32; 3],
    pub roughness: f32,
    pub emission: f32,
}

/// `Triangle {a, b, c, p_albedo_at, p_roughness_at, p_emission_at}` (shapes/mesh.rs:15-23)
#[repr(C)]
#[derive(Clone, Copy, Debug, Default)]
pub struct rt_triangle {
    pub a: [f32; 3],
    pub b: [f32; 3],
    pub c: [f32; 3],
    pub albedo: [f32; 3],
    pub roughness: f32,
    pub emission: f32,
}

/// `RenderMeta` + `division_no` (lib.rs:11-15,25-30) + the literals of main.rs:39-51 (0 = the reference's value)
#[repr(C)]
#[derive(Clone, Copy, Debug, Default)]
pub struct rt_params {
    pub width: u32,
    pub height: u32,
    pub divisions: u32,
    pub division_no: u32,
    pub spp: u32,
    pub max_bounces: u32,
    pub seed: u64,
    pub cam_origin: [f32; 3],
    pub aperture: f32,
    pub focus_distance: f32,
    pub field_of_view: f32,
    pub focal_length: f32,
    pub intersector: u32,
    pub collect_counters: u32,
    /// `RT_PARAM_*`: fields whose zero is a value, not "the reference's literal"
    pub flags: u32,
}
pub const RT_PARAM_MAX_BOUNCES_EXPLICIT: u32 = 1;
pub const RT_PARAM_APERTURE_EXPLICIT: u32 = 2;

#[repr(C)]
#[derive(Clone, Copy, Debug, Default)]
pub struct rt_stats {
    pub rays: u64,
    pub primary: u64,
    pub slab_tests: u64,
    pub sphere_tests: u64,
    pub sphere_exact: u64,
    pub sphere_hits: u64,
    pub tri_tests: u64,
    pub tri_stage: [u64; 3],
    pub tri_hits: u64,
    pub shades_sphere: u64,
    pub shades_tri: u64,
    pub emissive: u64,
    pub sky: u64,
    pub active_lane_iters: u64,
    pub total_lane_iters: u64,
    pub kernel_ms: f32,
    pub total_ms: f32,
    pub intersector_used: u32,
    pub kernel_launches: u32,
    pub grid_ctas: u32,
    pub cta_threads: u32,
    pub ctas_per_sm: u32,
    pub scene_in_smem: u32,
    pub dyn_smem_bytes: u32,
    pub redo_pixels: u32,
}

extern "C" {
    pub fn rt_abi_version() -> c_int;
    pub fn rt_struct_sizes(out: *mut usize);
    pub fn rt_init(device: c_int, out: *mut *mut rt_ctx) -> c_int;
    pub fn rt_shutdown(ctx: *mut rt_ctx);
    pub fn rt_last_error(ctx: *const rt_ctx) -> *const c_char;
    pub fn rt_scene_create(
        ctx: *mut rt_ctx,
        spheres: *const rt_sphere,
        n_spheres: u32,
        triangles: *const rt_triangle,
        n_triangles: u32,
        world_index: *const u32,
        out: *mut *mut rt_scene,
    ) -> c_int;
    pub fn rt_scene_destroy(ctx: *mut rt_ctx, scene: *mut rt_scene);
    pub fn rt_scene_update(
        ctx: *mut rt_ctx,
        scene: *mut rt_scene,
        spheres: *const rt_sphere,
        n_spheres: u32,
        triangles: *const rt_triangle,
        n_triangles: u32,
    ) -> c_int;
    pub fn rt_render_division(
        ctx: *mut rt_ctx,
        scene: *const rt_scene,
        params: *const rt_params,
        out_rgb: *mut u8,
        out_len: usize,
        stats: *mut rt_stats,
    ) -> c_int;
    pub fn rt_render_divisions(
        ctx: *mut rt_ctx,
        scene: *const rt_scene,
        params: *const rt_params,
        division_nos: *const u32,
        n: u32,
        out_rgb: *mut u8,
        out_len: usize,
        stats: *mut rt_stats,
    ) -> c_int;
    pub fn rt_render_frame(
        ctx: *mut rt_ctx,
        scene: *const rt_scene,
        params: *const rt_params,
        out_rgb: *mut u8,
        out_len: usize,
        stats: *mut rt_stats,
    ) -> c_int;
    pub fn rt_scene_wait_ready(ctx: *mut rt_ctx, scene: *const rt_scene) -> c_int;
    pub fn rt_render_frame_multi(
        ctxs: *const *mut rt_ctx,
        scenes: *const *const rt_scene,
        n: u32,
        params: *const rt_params,
        out_rgb: *mut u8,
        out_len: usize,
        stats: *mut rt_stats,
    ) -> c_int;
    pub fn rt_jpeg_bound(width: u32, height: u32) -> usize;
    pub fn rt_jpeg_encode(
        ctx: *mut rt_ctx,
        rgb: *const u8,
        width: u32,
        height: u32,
        quality: u32,
        out: *mut u8,
        out_cap: usize,
        out_len: *mut usize,
        ms_out: *mut f32,
    ) -> c_int;
    pub fn rt_render_frame_jpeg(
        ctxs: *const *mut rt_ctx,
        scenes: *const *const rt_scene,
        n: u32,
        params: *const rt_params,
        quality: u32,
        out: *mut u8,
        out_cap: usize,
        out_len: *mut usize,
        stats: *mut rt_stats,
    ) -> c_int;
    pub fn rt_world_json_max_objects(len: usize) -> usize;
    pub fn rt_world_parse_json(
        ctx: *mut rt_ctx,
        text: *const c_char,
        len: usize,
        spheres: *mut rt_sphere,
        triangles: *mut rt_triangle,
        world_index: *mut u32,
        cap: usize,
        n_spheres: *mut u32,
        n_triangles: *mut u32,
        consumed: *mut usize,
    ) -> c_int;
    pub fn rt_slice_json_bound(rows: u32, width: u32) -> usize;
    pub fn rt_obj_max_triangles(obj_size: usize) -> usize;
    pub fn rt_obj_build_world(
        ctx: *mut rt_ctx,
        body: *const u8,
        len: usize,
        obj_size: usize,
        triangles: *mut rt_triangle,
        cap: usize,
        n_triangles: *mut u32,
    ) -> c_int;
    pub fn rt_render_divisions_json(
        ctx: *mut rt_ctx,
        scene: *const rt_scene,
        params: *const rt_params,
        division_nos: *const u32,
        n: u32,
        id: *const c_char,
        out: *mut u8,
        out_cap: usize,
        out_lens: *mut usize,
        stats: *mut rt_stats,
    ) -> c_int;
    pub fn rt_render_tiles_device(
        ctx: *mut rt_ctx,
        scene: *const rt_scene,
        params: *const rt_params,
        tile_rank: u32,
        tile_ranks: u32,
        frame_dev: *mut c_void,
        sync: c_int,
        stats: *mut rt_stats,
    ) -> c_int;
    pub fn rt_accum_create(ctx: *mut rt_ctx, params: *const rt_params, out: *mut *mut rt_accum) -> c_int;
    pub fn rt_accum_destroy(ctx: *mut rt_ctx, acc: *mut rt_accum);
    pub fn rt_accum_reset(ctx: *mut rt_ctx, acc: *mut rt_accum, params: *const rt_params) -> c_int;
    pub fn rt_accum_samples(acc: *const rt_accum, samples_out: *mut u32) -> c_int;
    pub fn rt_render_samples(
        ctx: *mut rt_ctx,
        scene: *const rt_scene,
        acc: *mut rt_accum,
        n_samples: u32,
        out_rgb: *mut u8,
        out_len: usize,
        stats: *mut rt_stats,
    ) -> c_int;
    pub fn rt_accum_read_linear(ctx: *mut rt_ctx, acc: *const rt_accum, out: *mut f32, out_len: usize) -> c_int;
    pub fn rt_render_samples_multi(
        ctxs: *const *mut rt_ctx,
        scenes: *const *const rt_scene,
        accs: *const *mut rt_accum,
        n: u32,
        n_samples: u32,
        out_rgb: *mut u8,
        out_len: usize,
        stats: *mut rt_stats,
    ) -> c_int;
}

/// Error of any call: the negative `rt_status` and the library's message.
#[derive(Debug)]
pub struct Error {
    pub status: i32,
    pub message: String,
}
impl std::fmt::Display for Error {
    fn fmt(&self, f: &mut std::fmt::Formatter<'_>) -> std::fmt::Result {
        write!(f, "rt_b200 error {}: {}", self.status, self.message)
    }
}
impl std::error::Error for Error {}

/// One GPU + one stream.  `!Sync`: calls on a context are serialised by the owner, exactly like the
/// reference's single worker thread (main.rs:34-35,160).
pub struct Context {
    raw: *mut rt_ctx,
}
unsafe impl Send for Context {}

/// A world uploaded to the GPU (replaces `req.world` + `BVH::build`, main.rs:60-61).
pub struct Scene<'c> {
    ctx: &'c Context,
    raw: *mut rt_scene,
}

/// Resumable per-pixel sample chains of one band (`rt_accum`): chunks rendered with `render` add up, byte for byte, to
/// `render_division` at the cumulative sample count.
pub struct Accum<'c> {
    ctx: &'c Context,
    raw: *mut rt_accum,
    len: usize,
}

impl Context {
    pub fn new(device: i32) -> Result<Self, Error> {
        let mut sizes = [0usize; 4];
        unsafe { rt_struct_sizes(sizes.as_mut_ptr()) };
        assert_eq!(
            sizes,
            [
                std::mem::size_of::<rt_sphere>(),
                std::mem::size_of::<rt_triangle>(),
                std::mem::size_of::<rt_params>(),
                std::mem::size_of::<rt_stats>()
            ],
            "struct layout mismatch between librt_b200.so and this crate"
        );
        let mut raw = ptr::null_mut();
        let rc = unsafe { rt_init(device, &mut raw) };
        if rc != 0 {
            return Err(Error { status: rc, message: last_error(ptr::null()) });
        }
        Ok(Context { raw })
    }

    fn check(&self, rc: c_int) -> Result<(), Error> {
        if rc == 0 {
            Ok(())
        } else {
            Err(Error { status: rc, message: last_error(self.raw) })
        }
    }

    /// `world_index[i]` = position of primitive i (spheres first, then triangles) in the `Vec<Object>`.
    pub fn scene(&self, spheres: &[rt_sphere], triangles: &[rt_triangle], world_index: Option<&[u32]>) -> Result<Scene<'_>, Error> {
        if let Some(w) = world_index {
            // the C side reads n_spheres + n_triangles entries
            if w.len() != spheres.len() + triangles.len() {
                return Err(Error {
                    status: -1,
                    message: format!("world_index has {} entries for {} primitives", w.len(), spheres.len() + triangles.len()),
                });
            }
        }
        let mut raw = ptr::null_mut();
        let wi = world_index.map_or(ptr::null(), |w| w.as_ptr());
        let rc = unsafe {
            rt_scene_create(self.raw, spheres.as_ptr(), spheres.len() as u32, triangles.as_ptr(), triangles.len() as u32, wi, &mut raw)
        };
        self.check(rc)?;
        Ok(Scene { ctx: self, raw })
    }

    /// Band `params.division_no` → `(height/divisions) * width * 3` RGB bytes, row 0 = top of the band:
    /// the `img_buff` of main.rs:53-83.
    pub fn render_division(&self, scene: &Scene<'_>, params: &rt_params) -> Result<Vec<u8>, Error> {
        let div = params.divisions.max(1);
        let len = (params.height / div) as usize * params.width as usize * 3;
        let mut out = vec![0u8; len];
        let rc = unsafe { rt_render_division(self.raw, scene.raw, params, out.as_mut_ptr(), out.len(), ptr::null_mut()) };
        self.check(rc)?;
        Ok(out)
    }

    /// Bands `division_nos` of one job in one launch (`params.division_no` is ignored): band `division_nos[k]` is
    /// `out[k * rows * width * 3..][..rows * width * 3]`, the bytes `render_division` gives for it.
    pub fn render_divisions(&self, scene: &Scene<'_>, params: &rt_params, division_nos: &[u32]) -> Result<Vec<u8>, Error> {
        let div = params.divisions.max(1);
        let len = division_nos.len() * (params.height / div) as usize * params.width as usize * 3;
        let mut out = vec![0u8; len];
        let rc = unsafe {
            rt_render_divisions(self.raw, scene.raw, params, division_nos.as_ptr(), division_nos.len() as u32, out.as_mut_ptr(),
                                out.len(), ptr::null_mut())
        };
        self.check(rc)?;
        Ok(out)
    }

    /// The `world` of a RenderInfo body (the raw JSON text of the array) parsed on the GPU: spheres, triangles and the
    /// world position of each (spheres first), what `Vec<Object>` holds.  `None` when the text is outside the device
    /// grammar (serde's own layout of `Object`, numbers of at most 19 digits): deserialize `Vec<Object>` then, which
    /// decides whether the body is valid.
    pub fn parse_world_json(&self, text: &str) -> Option<(Vec<rt_sphere>, Vec<rt_triangle>, Vec<u32>)> {
        let cap = unsafe { rt_world_json_max_objects(text.len()) };
        let (mut sp, mut tr, mut wi) = (Vec::with_capacity(cap), Vec::with_capacity(cap), Vec::with_capacity(cap));
        let (mut ns, mut nt, mut used) = (0u32, 0u32, 0usize);
        let rc = unsafe {
            rt_world_parse_json(self.raw, text.as_ptr() as *const c_char, text.len(), sp.as_mut_ptr(), tr.as_mut_ptr(),
                                wi.as_mut_ptr(), cap, &mut ns, &mut nt, &mut used)
        };
        // a text with more after the array is not a world value (serde's RawValue holds exactly the value)
        if rc != 0 || !text[used..].trim_matches(|c| matches!(c, ' ' | '\t' | '\n' | '\r')).is_empty() {
            return None;
        }
        unsafe {
            sp.set_len(ns as usize);
            tr.set_len(nt as usize);
            wi.set_len((ns + nt) as usize);
        }
        Some((sp, tr, wi))
    }

    /// The controller's `/upload` body (`body[..obj_size]` the OBJ, the rest the MTL) built into its world on the GPU:
    /// the triangles `obj::build_world` returns (obj.rs:10-53), in its order.  `None` when the body is outside the device
    /// grammar, which includes every body `obj::build_world` rejects: call it then, which decides whether the body is
    /// valid.
    pub fn build_world_obj(&self, body: &[u8], obj_size: usize) -> Option<Vec<rt_triangle>> {
        if obj_size > body.len() {
            return None;
        }
        let cap = unsafe { rt_obj_max_triangles(obj_size) };
        let mut tr = Vec::with_capacity(cap);
        let mut n = 0u32;
        let rc = unsafe { rt_obj_build_world(self.raw, body.as_ptr(), body.len(), obj_size, tr.as_mut_ptr(), cap, &mut n) };
        if rc != 0 {
            return None;
        }
        unsafe { tr.set_len(n as usize) };
        Some(tr)
    }

    /// `render_divisions`, then each band as the ImageSlice body the slave POSTs to /result, written on the device: body
    /// k is `serde_json::to_vec(&ImageSlice { division_no: division_nos[k], image, id })`.  `id`: the hyphenated
    /// lowercase uuid (`Uuid::to_string`).
    pub fn render_divisions_json(&self, scene: &Scene<'_>, params: &rt_params, division_nos: &[u32], id: &str)
                                 -> Result<Vec<Vec<u8>>, Error> {
        let rows = params.height / params.divisions.max(1);
        let mut out = vec![0u8; division_nos.len() * unsafe { rt_slice_json_bound(rows, params.width) }];
        let mut lens = vec![0usize; division_nos.len()];
        let id = std::ffi::CString::new(id).map_err(|_| Error { status: -1, message: "id holds a NUL".into() })?;
        let rc = unsafe {
            rt_render_divisions_json(self.raw, scene.raw, params, division_nos.as_ptr(), division_nos.len() as u32,
                                     id.as_ptr(), out.as_mut_ptr(), out.len(), lens.as_mut_ptr(), ptr::null_mut())
        };
        self.check(rc)?;
        let mut at = 0;
        Ok(lens.iter().map(|&n| { let b = out[at..at + n].to_vec(); at += n; b }).collect())
    }

    /// Baseline JPEG of an RGB8 frame (`height * width * 3` bytes, row 0 on top), encoded on this context's GPU: the
    /// bytes libjpeg writes with its defaults at `quality` (1..100), i.e. the controller's JPEG(90) at 90.
    pub fn encode_jpeg(&self, rgb: &[u8], width: u32, height: u32, quality: u32) -> Result<Vec<u8>, Error> {
        assert_eq!(rgb.len(), width as usize * height as usize * 3, "rgb must hold height * width * 3 bytes");
        let mut out = vec![0u8; unsafe { rt_jpeg_bound(width, height) }];
        let mut len = 0usize;
        let rc = unsafe {
            rt_jpeg_encode(self.raw, rgb.as_ptr(), width, height, quality, out.as_mut_ptr(), out.len(), &mut len, ptr::null_mut())
        };
        self.check(rc)?;
        out.truncate(len);
        Ok(out)
    }

    /// The whole frame of `render_frame` as JPEG bytes, encoded on the device where it was rendered: equal to
    /// `encode_jpeg(&render_frame(..)?, ..)` without the RGB frame crossing to the host.
    pub fn render_frame_jpeg(&self, scene: &Scene<'_>, params: &rt_params, quality: u32) -> Result<Vec<u8>, Error> {
        render_frame_jpeg(&[self], &[scene], params, quality)
    }

    /// Sample state of the band `params` selects (`params.spp` is ignored), every pixel at sample 0.
    pub fn accum(&self, params: &rt_params) -> Result<Accum<'_>, Error> {
        let div = params.divisions.max(1);
        let mut raw = ptr::null_mut();
        self.check(unsafe { rt_accum_create(self.raw, params, &mut raw) })?;
        Ok(Accum { ctx: self, raw, len: (params.height / div) as usize * params.width as usize * 3 })
    }
}

impl Scene<'_> {
    /// Replaces the world with one of the same shape (as many spheres and triangles as created; the creation's
    /// `world_index` still applies).  Later renders are byte-identical to those of a scene created from the new world;
    /// an `Accum` with samples of the old world needs `reset`.  On an error other than status -4 (CUDA) the scene still
    /// holds the old world; after -4 drop it.
    pub fn update(&mut self, spheres: &[rt_sphere], triangles: &[rt_triangle]) -> Result<(), Error> {
        let rc = unsafe {
            rt_scene_update(self.ctx.raw, self.raw, spheres.as_ptr(), spheres.len() as u32, triangles.as_ptr(), triangles.len() as u32)
        };
        self.ctx.check(rc)
    }
}

impl Accum<'_> {
    /// Advances every pixel by `n_samples` and returns the band as it now stands: the bytes of `render_division` at
    /// `spp = self.samples()`.
    pub fn render(&mut self, scene: &Scene<'_>, n_samples: u32) -> Result<Vec<u8>, Error> {
        let mut out = vec![0u8; self.len];
        let rc = unsafe { rt_render_samples(self.ctx.raw, scene.raw, self.raw, n_samples, out.as_mut_ptr(), out.len(), ptr::null_mut()) };
        self.ctx.check(rc)?;
        Ok(out)
    }

    /// Back to sample 0, optionally with new params of the same size and band.
    pub fn reset(&mut self, params: Option<&rt_params>) -> Result<(), Error> {
        let p = params.map_or(ptr::null(), |p| p as *const rt_params);
        self.ctx.check(unsafe { rt_accum_reset(self.ctx.raw, self.raw, p) })
    }

    pub fn samples(&self) -> u32 {
        let mut n = 0u32;
        unsafe { rt_accum_samples(self.raw, &mut n) };
        n
    }
}

/// One frame over several GPUs from this process (`rt_render_frame_multi`): `ctxs[i]` renders rank i's share of the
/// 8x4 tiles of `scenes[i]` (the same world uploaded on that context) straight into `ctxs[0]`'s frame over NVLink; the
/// frame streams to the returned buffer while it renders.  This is the controller's fan-out + stitch
/// (ray-tracer-controller/src/main.rs:47-75,109-119) without HTTP.
pub fn render_frame_multi(ctxs: &[&Context], scenes: &[&Scene<'_>], params: &rt_params) -> Result<Vec<u8>, Error> {
    assert!(!ctxs.is_empty() && ctxs.len() == scenes.len(), "one scene per context");
    let c: Vec<*mut rt_ctx> = ctxs.iter().map(|c| c.raw).collect();
    let s: Vec<*const rt_scene> = scenes.iter().map(|s| s.raw as *const rt_scene).collect();
    let mut out = vec![0u8; params.height as usize * params.width as usize * 3];
    let rc = unsafe { rt_render_frame_multi(c.as_ptr(), s.as_ptr(), c.len() as u32, params, out.as_mut_ptr(), out.len(), ptr::null_mut()) };
    ctxs[0].check(rc)?;
    Ok(out)
}

/// The frame of `render_frame_multi` (or of `Context::render_frame` for one context) as JPEG bytes at `quality`,
/// encoded on `ctxs[0]`'s GPU where the frame lies (`rt_render_frame_jpeg`).  What a controller returns from `/poll`.
pub fn render_frame_jpeg(ctxs: &[&Context], scenes: &[&Scene<'_>], params: &rt_params, quality: u32) -> Result<Vec<u8>, Error> {
    assert!(!ctxs.is_empty() && ctxs.len() == scenes.len(), "one scene per context");
    let c: Vec<*mut rt_ctx> = ctxs.iter().map(|c| c.raw).collect();
    let s: Vec<*const rt_scene> = scenes.iter().map(|s| s.raw as *const rt_scene).collect();
    let mut out = vec![0u8; unsafe { rt_jpeg_bound(params.width, params.height) }];
    let mut len = 0usize;
    let rc = unsafe {
        rt_render_frame_jpeg(c.as_ptr(), s.as_ptr(), c.len() as u32, params, quality, out.as_mut_ptr(), out.len(), &mut len,
                             ptr::null_mut())
    };
    ctxs[0].check(rc)?;
    out.truncate(len);
    Ok(out)
}

/// One progressive frame over several GPUs (`rt_render_samples_multi`): `accs[i]` (a whole-frame `Accum` of `ctxs[i]`)
/// holds the chains of rank i's tiles of `scenes[i]`; every pixel advances by `n_samples` and the returned frame is the
/// bytes of `render_frame_multi` at `spp = accs[0].samples()`.  On an error no accum moves.
pub fn render_samples_multi(ctxs: &[&Context], scenes: &[&Scene<'_>], accs: &mut [&mut Accum<'_>], n_samples: u32) -> Result<Vec<u8>, Error> {
    assert!(!ctxs.is_empty() && ctxs.len() == scenes.len() && ctxs.len() == accs.len(), "one scene and one accum per context");
    let c: Vec<*mut rt_ctx> = ctxs.iter().map(|c| c.raw).collect();
    let s: Vec<*const rt_scene> = scenes.iter().map(|s| s.raw as *const rt_scene).collect();
    let a: Vec<*mut rt_accum> = accs.iter().map(|a| a.raw).collect();
    let mut out = vec![0u8; accs[0].len];
    let rc = unsafe {
        rt_render_samples_multi(c.as_ptr(), s.as_ptr(), a.as_ptr(), c.len() as u32, n_samples, out.as_mut_ptr(), out.len(), ptr::null_mut())
    };
    ctxs[0].check(rc)?;
    Ok(out)
}

impl Drop for Context {
    fn drop(&mut self) {
        unsafe { rt_shutdown(self.raw) }
    }
}
impl Drop for Accum<'_> {
    fn drop(&mut self) {
        unsafe { rt_accum_destroy(self.ctx.raw, self.raw) }
    }
}
impl Drop for Scene<'_> {
    fn drop(&mut self) {
        unsafe { rt_scene_destroy(self.ctx.raw, self.raw) }
    }
}

fn last_error(ctx: *const rt_ctx) -> String {
    unsafe { CStr::from_ptr(rt_last_error(ctx)).to_string_lossy().into_owned() }
}
