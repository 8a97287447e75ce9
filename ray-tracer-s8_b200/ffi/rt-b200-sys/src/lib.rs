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
    pub fn rt_render_division(
        ctx: *mut rt_ctx,
        scene: *const rt_scene,
        params: *const rt_params,
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

    /// Sample state of the band `params` selects (`params.spp` is ignored), every pixel at sample 0.
    pub fn accum(&self, params: &rt_params) -> Result<Accum<'_>, Error> {
        let div = params.divisions.max(1);
        let mut raw = ptr::null_mut();
        self.check(unsafe { rt_accum_create(self.raw, params, &mut raw) })?;
        Ok(Accum { ctx: self, raw, len: (params.height / div) as usize * params.width as usize * 3 })
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
