//! gpu.rs -- the `gpu` module a vecchio maintainer would add next to src/main.rs to call the
//! B200 library (include/vecchio_gpu.h, libvecchio_gpu.so) instead of the rayon sample loop.
//!
//! STATUS: SOURCE ONLY.  This image has no rustc/cargo, so this file has never been compiled or
//! run; the C ABI it binds is exercised by the Python ctypes harness and the C++ front end
//! instead (tests/, vecchio_b200/host/).  See INTEGRATION.md for the three edits to the reference
//! (mod gpu; one `lower()` method per trait; the call in main()).
//!
//! Layouts mirror include/vecchio_gpu.h field by field (`#[repr(C)]`); Vec3/Camera/Ray of the
//! reference are NOT repr(C) (src/vec3.rs:3-8, src/main.rs:31-36,56-68) and are copied.
#![allow(non_camel_case_types, dead_code)]

use std::collections::HashMap;
use std::ffi::CStr;
use std::os::raw::{c_char, c_int, c_void};
use std::sync::Arc;

use crate::hittable::{Hittable, HittableSS};                    // the traits must be in scope to call `lower` on the trait objects
use crate::material::{Material, MaterialSS, Texture, TextureSS};
use crate::vec3::Vec3;

/// `Vec3` is not `repr(C)` (src/vec3.rs:3-8): copied field by field.
pub fn v3(v: Vec3) -> [f32; 3] { [v.x, v.y, v.z] }

pub type vk_ref = u32; // (type << 28) | index ; 0 == none
pub const VK_API_VERSION: u32 = 1;
pub const VK_T_NODE: u32 = 1;
pub const VK_T_SPHERE: u32 = 2;
pub const VK_T_MSPHERE: u32 = 3;
pub const VK_T_RECT: u32 = 4;
pub const VK_T_BOX: u32 = 5;
pub const VK_T_XFORM: u32 = 6;
pub const VK_T_MEDIUM: u32 = 7;
pub const VK_RECT_FLIP: u32 = 0x100;
pub const VK_X_TRANSLATE: u32 = 0;
pub const VK_X_ROTATE_X: u32 = 1;
pub const VK_X_ROTATE_Y: u32 = 2;
pub const VK_X_ROTATE_Z: u32 = 3;
pub const VK_X_FLIP: u32 = 4;
pub const VK_M_LAMBERTIAN: u32 = 0;
pub const VK_M_METAL: u32 = 1;
pub const VK_M_DIELECTRIC: u32 = 2;
pub const VK_M_DIFFUSE_LIGHT: u32 = 3;
pub const VK_M_ISOTROPIC: u32 = 4;
pub const VK_M_SPECDIFFUSE: u32 = 5;
pub const VK_TEX_SOLID: u32 = 0;
pub const VK_TEX_CHECKER: u32 = 1;
pub const VK_TEX_IMAGE: u32 = 2;
pub const VK_TEX_NOISE: u32 = 3;
pub const fn vk_mkref(t: u32, i: u32) -> vk_ref { (t << 28) | (i & 0x0FFF_FFFF) }

#[repr(C)] #[derive(Clone, Copy, Default)] pub struct vk_node { pub bb_min: [f32; 3], pub left: vk_ref, pub bb_max: [f32; 3], pub right: vk_ref }
#[repr(C)] #[derive(Clone, Copy, Default)] pub struct vk_sphere { pub center: [f32; 3], pub radius: f32 }
#[repr(C)] #[derive(Clone, Copy, Default)] pub struct vk_msphere { pub center0: [f32; 3], pub radius: f32, pub center1: [f32; 3], pub time0: f32, pub time1: f32, pub mat: u32, pub _pad: [u32; 2] }
#[repr(C)] #[derive(Clone, Copy, Default)] pub struct vk_rect { pub c0: f32, pub c1: f32, pub d0: f32, pub d1: f32, pub k: f32, pub axes: u32, pub mat: u32, pub _pad: u32 }
#[repr(C)] #[derive(Clone, Copy, Default)] pub struct vk_box { pub box_min: [f32; 3], pub mat: u32, pub box_max: [f32; 3], pub _pad: u32 }
#[repr(C)] #[derive(Clone, Copy, Default)] pub struct vk_xform { pub kind: u32, pub child: vk_ref, pub _pad0: [u32; 2], pub a: f32, pub b: f32, pub c: f32, pub _pad1: u32 }
#[repr(C)] #[derive(Clone, Copy, Default)] pub struct vk_medium { pub boundary: vk_ref, pub neg_inv_density: f32, pub mat: u32, pub _pad: u32 }
#[repr(C)] #[derive(Clone, Copy, Default)] pub struct vk_material { pub type_: u32, pub tex: u32, pub param: f32, pub aux: u32 }
#[repr(C)] #[derive(Clone, Copy, Default)] pub struct vk_texture { pub type_: u32, pub w: [u32; 3] } // union payload as 3 words (f32::to_bits for SOLID)
#[repr(C)] #[derive(Clone, Copy)] pub struct vk_perlin { pub ranvec: [[f32; 3]; 256], pub perm_x: [u8; 256], pub perm_y: [u8; 256], pub perm_z: [u8; 256] }

#[repr(C)]
pub struct vk_scene_desc {
    pub api_version: u32, pub root: vk_ref,
    pub nodes: *const vk_node, pub n_nodes: u32,
    pub spheres: *const vk_sphere, pub sphere_mat: *const u32, pub n_spheres: u32,
    pub mspheres: *const vk_msphere, pub n_mspheres: u32,
    pub rects: *const vk_rect, pub n_rects: u32,
    pub boxes: *const vk_box, pub n_boxes: u32,
    pub xforms: *const vk_xform, pub n_xforms: u32,
    pub media: *const vk_medium, pub n_media: u32,
    pub lights: *const vk_ref, pub n_lights: u32,
    pub materials: *const vk_material, pub n_materials: u32,
    pub textures: *const vk_texture, pub n_textures: u32,
    pub texels: *const u8, pub n_texel_bytes: u64,
    pub perlins: *const vk_perlin, pub n_perlins: u32,
}
#[repr(C)] #[derive(Clone, Copy, Default)]
pub struct vk_camera { pub origin: [f32; 3], pub lower_left_corner: [f32; 3], pub horizontal: [f32; 3], pub vertical: [f32; 3],
                       pub u: [f32; 3], pub v: [f32; 3], pub w: [f32; 3], pub lens_radius: f32, pub time0: f32, pub time1: f32 }
#[repr(C)] #[derive(Clone, Copy, Default)]
pub struct vk_render_params { pub width: u32, pub height: u32, pub spp: u32, pub spp_begin: u32, pub spp_count: u32, pub max_depth: u32,
                              pub seed: u64, pub background: [f32; 3], pub variant: u32, pub flags: u32 }
#[repr(C)] #[derive(Clone, Copy, Default)]
pub struct vk_stats { pub paths: u64, pub rays: u64, pub dropped_samples: u64, pub ms_kernels: f32, pub ms_total: f32,
                      pub variant: u32, pub launches: u32, pub node_visits: u64, pub prim_tests: u64 }
#[repr(C)] pub struct vk_ctx { _private: [u8; 0] }
#[repr(C)] #[derive(Clone, Copy, Default, PartialEq)]
pub struct vk_adaptive_target { pub spp: u32, pub min_spp: u32, pub max_error: f32 }
#[repr(C)] pub struct vk_adaptive_session { _private: [u8; 0] }

#[link(name = "vecchio_gpu")]
extern "C" {
    pub fn vk_create(device: c_int, out: *mut *mut vk_ctx) -> c_int;
    pub fn vk_destroy(ctx: *mut vk_ctx);
    pub fn vk_last_error(ctx: *const vk_ctx) -> *const c_char;
    pub fn vk_scene_upload(ctx: *mut vk_ctx, scene: *const vk_scene_desc) -> c_int;
    pub fn vk_render(ctx: *mut vk_ctx, cam: *const vk_camera, params: *const vk_render_params,
                     out_rgb: *mut f32, out_sumsq: *mut f32, stats: *mut vk_stats) -> c_int;
    pub fn vk_render_rgb8(ctx: *mut vk_ctx, cam: *const vk_camera, params: *const vk_render_params,
                          out_rgb8: *mut u8, stats: *mut vk_stats) -> c_int;
    pub fn vk_render_device(ctx: *mut vk_ctx, cam: *const vk_camera, params: *const vk_render_params,
                            d_sum: *mut f32, d_sumsq: *mut f32, stats: *mut vk_stats) -> c_int;
    pub fn vk_finalize_device(ctx: *mut vk_ctx, d_sum: *const f32, d_rgb: *mut f32, n_floats: usize, spp: u32) -> c_int;
    pub fn vk_set_stream(ctx: *mut vk_ctx, stream: *mut c_void) -> c_int;
    pub fn vk_flush_stats(ctx: *mut vk_ctx, stats: *mut vk_stats) -> c_int;
    // K cameras in one launch: frame f uses cams[f] and seed + f, and equals vk_render / vk_render_rgb8 of that camera bit for bit
    // on the same kernel (AUTO decides on the batch's path count; the render build's kernels round differently)
    pub fn vk_render_frames(ctx: *mut vk_ctx, cams: *const vk_camera, n_frames: u32, params: *const vk_render_params,
                            out_rgb: *mut f32, stats: *mut vk_stats) -> c_int;
    pub fn vk_render_frames_rgb8(ctx: *mut vk_ctx, cams: *const vk_camera, n_frames: u32, params: *const vk_render_params,
                                 out_rgb8: *mut u8, stats: *mut vk_stats) -> c_int;
    // feature buffers for a denoiser: first-hit albedo, normal, depth and coverage of the render's own camera rays for samples
    // 0 .. aov_spp-1 (the header states each plane); every output nullable, at least one non-null
    pub fn vk_render_aov(ctx: *mut vk_ctx, cams: *const vk_camera, n_frames: u32, params: *const vk_render_params, aov_spp: u32,
                         out_albedo: *mut f32, out_normal: *mut f32, out_depth: *mut f32, out_coverage: *mut f32,
                         stats: *mut vk_stats) -> c_int;
    // adaptive sampling: passes of pass_spp samples until a pixel's displayed noise is <= max_error (8-bit steps) or spp;
    // a pixel that stopped at n samples equals vk_render with spp = n on the same kernel (the header states the rule)
    pub fn vk_render_adaptive(ctx: *mut vk_ctx, cam: *const vk_camera, params: *const vk_render_params, pass_spp: u32, max_error: f32,
                              out_rgb: *mut f32, out_spp: *mut u32, stats: *mut vk_stats) -> c_int;
    pub fn vk_render_adaptive_rgb8(ctx: *mut vk_ctx, cam: *const vk_camera, params: *const vk_render_params, pass_spp: u32,
                                   max_error: f32, out_rgb8: *mut u8, out_spp: *mut u32, stats: *mut vk_stats) -> c_int;
    // adaptive sampling of K cameras: every pass one launch over the active pixels of all frames; frame f (cams[f], seed + f)
    // and its counts equal vk_render_adaptive of that camera (bit for bit with VK_FLAG_STRICT_MATH; the header states the render build)
    pub fn vk_render_frames_adaptive(ctx: *mut vk_ctx, cams: *const vk_camera, n_frames: u32, params: *const vk_render_params,
                                     pass_spp: u32, max_error: f32, out_rgb: *mut f32, out_spp: *mut u32, stats: *mut vk_stats) -> c_int;
    pub fn vk_render_frames_adaptive_rgb8(ctx: *mut vk_ctx, cams: *const vk_camera, n_frames: u32, params: *const vk_render_params,
                                          pass_spp: u32, max_error: f32, out_rgb8: *mut u8, out_spp: *mut u32, stats: *mut vk_stats) -> c_int;
    // adaptive sessions: the state of an adaptive render kept between calls, moved by tightening targets; each refine ends
    // bit for bit where a fresh session refined once to that target would (the header states the rule and the refusals)
    pub fn vk_adaptive_begin(ctx: *mut vk_ctx, cams: *const vk_camera, n_frames: u32, params: *const vk_render_params, pass_spp: u32,
                             out: *mut *mut vk_adaptive_session) -> c_int;
    pub fn vk_adaptive_refine(session: *mut vk_adaptive_session, target: *const vk_adaptive_target, stats: *mut vk_stats) -> c_int;
    pub fn vk_adaptive_read(session: *mut vk_adaptive_session, out_rgb: *mut f32, out_spp: *mut u32, out_error: *mut f32) -> c_int;
    pub fn vk_adaptive_read_rgb8(session: *mut vk_adaptive_session, out_rgb8: *mut u8, out_spp: *mut u32, out_error: *mut f32) -> c_int;
    pub fn vk_adaptive_export(session: *mut vk_adaptive_session, sums: *mut i64, squares: *mut u64, counts: *mut u32,
                              reached: *mut vk_adaptive_target) -> c_int;
    pub fn vk_adaptive_import(session: *mut vk_adaptive_session, sums: *const i64, squares: *const u64, counts: *const u32,
                              reached: *const vk_adaptive_target) -> c_int;
    pub fn vk_adaptive_variant(session: *const vk_adaptive_session) -> u32;
    pub fn vk_adaptive_destroy(session: *mut vk_adaptive_session);
    // a session over the pixels shard `shard` of n_shards owns ((g / VK_SHARD_RUN) mod n_shards == shard); the shards' exports
    // add up to the unsharded session's bit for bit
    pub fn vk_adaptive_begin_shard(ctx: *mut vk_ctx, cams: *const vk_camera, n_frames: u32, params: *const vk_render_params, pass_spp: u32,
                                   shard: u32, n_shards: u32, out: *mut *mut vk_adaptive_session) -> c_int;
    // one context over several GPUs of the node (samples split by global index, peer-memory reduce on devices[0])
    pub fn vk_multi_create(devices: *const c_int, n_devices: c_int, out: *mut *mut vk_multi) -> c_int;
    pub fn vk_multi_destroy(m: *mut vk_multi);
    pub fn vk_multi_last_error(m: *const vk_multi) -> *const c_char;
    pub fn vk_multi_scene_upload(m: *mut vk_multi, scene: *const vk_scene_desc) -> c_int;
    pub fn vk_multi_render(m: *mut vk_multi, cam: *const vk_camera, params: *const vk_render_params,
                           out_rgb: *mut f32, out_sumsq: *mut f32, stats: *mut vk_stats) -> c_int;
    pub fn vk_multi_render_rgb8(m: *mut vk_multi, cam: *const vk_camera, params: *const vk_render_params,
                                out_rgb8: *mut u8, stats: *mut vk_stats) -> c_int;
    pub fn vk_multi_render_frames_rgb8(m: *mut vk_multi, cams: *const vk_camera, n_frames: u32, params: *const vk_render_params,
                                       out_rgb8: *mut u8, stats: *mut vk_stats) -> c_int;
    pub fn vk_multi_render_aov(m: *mut vk_multi, cams: *const vk_camera, n_frames: u32, params: *const vk_render_params, aov_spp: u32,
                               out_albedo: *mut f32, out_normal: *mut f32, out_depth: *mut f32, out_coverage: *mut f32,
                               stats: *mut vk_stats) -> c_int;
    // adaptive sampling over several GPUs: device k renders shard k's pixels; every result equals the one-GPU call's bit for bit
    pub fn vk_multi_adaptive_begin(m: *mut vk_multi, cams: *const vk_camera, n_frames: u32, params: *const vk_render_params, pass_spp: u32,
                                   out: *mut *mut vk_multi_adaptive_session) -> c_int;
    pub fn vk_multi_adaptive_refine(session: *mut vk_multi_adaptive_session, target: *const vk_adaptive_target, stats: *mut vk_stats) -> c_int;
    pub fn vk_multi_adaptive_read(session: *mut vk_multi_adaptive_session, out_rgb: *mut f32, out_spp: *mut u32, out_error: *mut f32) -> c_int;
    pub fn vk_multi_adaptive_read_rgb8(session: *mut vk_multi_adaptive_session, out_rgb8: *mut u8, out_spp: *mut u32, out_error: *mut f32) -> c_int;
    pub fn vk_multi_adaptive_export(session: *mut vk_multi_adaptive_session, sums: *mut i64, squares: *mut u64, counts: *mut u32,
                                    reached: *mut vk_adaptive_target) -> c_int;
    pub fn vk_multi_adaptive_import(session: *mut vk_multi_adaptive_session, sums: *const i64, squares: *const u64, counts: *const u32,
                                    reached: *const vk_adaptive_target) -> c_int;
    pub fn vk_multi_adaptive_variant(session: *const vk_multi_adaptive_session) -> u32;
    pub fn vk_multi_adaptive_destroy(session: *mut vk_multi_adaptive_session);
    pub fn vk_multi_render_adaptive_rgb8(m: *mut vk_multi, cam: *const vk_camera, params: *const vk_render_params, pass_spp: u32,
                                         max_error: f32, out_rgb8: *mut u8, out_spp: *mut u32, stats: *mut vk_stats) -> c_int;
    pub fn vk_multi_render_frames_adaptive_rgb8(m: *mut vk_multi, cams: *const vk_camera, n_frames: u32, params: *const vk_render_params,
                                                pass_spp: u32, max_error: f32, out_rgb8: *mut u8, out_spp: *mut u32, stats: *mut vk_stats) -> c_int;
}
#[repr(C)] pub struct vk_multi { _private: [u8; 0] }
#[repr(C)] pub struct vk_multi_adaptive_session { _private: [u8; 0] }
pub const VK_SHARD_RUN: u32 = 32;

#[derive(Debug)]
pub enum GpuError { Unsupported(&'static str), Library(i32, String) }

/// Accumulates the flat arrays while the object graph is walked.  Shared `Arc`s are lowered once
/// (keyed by pointer), so the 400 boxes that share one material produce one material record.
#[derive(Default)]
pub struct Lowering {
    pub nodes: Vec<vk_node>, pub spheres: Vec<vk_sphere>, pub sphere_mat: Vec<u32>, pub mspheres: Vec<vk_msphere>,
    pub rects: Vec<vk_rect>, pub boxes: Vec<vk_box>, pub xforms: Vec<vk_xform>, pub media: Vec<vk_medium>,
    pub lights: Vec<vk_ref>, pub materials: Vec<vk_material>, pub textures: Vec<vk_texture>, pub texels: Vec<u8>,
    pub perlins: Vec<vk_perlin>,
    // allocation address -> record: Arc::as_ptr(..) as *const () as usize (one map per trait, one for flipped rects)
    pub memo_h: HashMap<usize, vk_ref>, pub memo_flip: HashMap<usize, vk_ref>, pub memo_m: HashMap<usize, u32>, pub memo_t: HashMap<usize, u32>,
}

impl Lowering {
    /// `h.lower(self)`, once per allocation: a sub-BVH under two wrappers, a rect that is both a world object
    /// (inside its FlipFace) and a light, come out as ONE record.  The C++ model of these three is
    /// `Lowering::hittable / material / texture` in vecchio_b200/host/vecchio.cpp.
    pub fn hittable(&mut self, h: &Arc<HittableSS>) -> Result<vk_ref, GpuError> {
        let key = Arc::as_ptr(h) as *const () as usize;
        if let Some(&r) = self.memo_h.get(&key) { return Ok(r); }
        let r = h.lower(self)?;
        self.memo_h.insert(key, r);
        Ok(r)
    }
    pub fn material(&mut self, m: &Arc<MaterialSS>) -> Result<u32, GpuError> {
        let key = Arc::as_ptr(m) as *const () as usize;
        if let Some(&i) = self.memo_m.get(&key) { return Ok(i); }
        let i = m.lower(self)?;
        self.memo_m.insert(key, i);
        Ok(i)
    }
    pub fn texture(&mut self, t: &Arc<TextureSS>) -> Result<u32, GpuError> {
        let key = Arc::as_ptr(t) as *const () as usize;
        if let Some(&i) = self.memo_t.get(&key) { return Ok(i); }
        let i = t.lower(self)?;
        self.memo_t.insert(key, i);
        Ok(i)
    }
    pub fn push_material(&mut self, type_: u32, tex: u32, param: f32, aux: u32) -> u32 {
        self.materials.push(vk_material { type_, tex, param, aux });
        (self.materials.len() - 1) as u32
    }
    pub fn push_texture(&mut self, type_: u32, w: [u32; 3]) -> u32 {
        self.textures.push(vk_texture { type_, w });
        (self.textures.len() - 1) as u32
    }
    pub fn push_xform(&mut self, kind: u32, child: vk_ref, a: f32, b: f32, c: f32) -> vk_ref {
        self.xforms.push(vk_xform { kind, child, _pad0: [0; 2], a, b, c, _pad1: 0 });
        vk_mkref(VK_T_XFORM, (self.xforms.len() - 1) as u32)
    }
}

/// The ONE method added to each of the reference's traits (they are otherwise opaque: no `Any`,
/// private fields).  The default reports the type as unsupported, so a user-defined Hittable makes
/// `render` fail loudly instead of being skipped:
///
/// ```ignore
/// // src/hittable.rs:33-42
/// pub trait Hittable { /* hit, bounding_box, pdf_value, random as before */
///     fn lower(&self, _b: &mut gpu::Lowering) -> Result<gpu::vk_ref, gpu::GpuError> {
///         Err(gpu::GpuError::Unsupported("Hittable"))
///     }
/// }
/// impl Hittable for Sphere {                      // src/hittable.rs:63
///     fn lower(&self, b: &mut gpu::Lowering) -> Result<gpu::vk_ref, gpu::GpuError> {
///         let mat = b.material(&self.material)?;  // memoised Material::lower -> index into b.materials
///         b.spheres.push(gpu::vk_sphere { center: gpu::v3(self.center), radius: self.radius });
///         b.sphere_mat.push(mat);
///         Ok(gpu::vk_mkref(gpu::VK_T_SPHERE, (b.spheres.len() - 1) as u32))
///     }
/// }
/// impl Hittable for BVHNode {                     // src/accel.rs:58
///     fn lower(&self, b: &mut gpu::Lowering) -> Result<gpu::vk_ref, gpu::GpuError> {
///         let i = b.nodes.len();                  // depth first, parent before children, left first
///         b.nodes.push(Default::default());
///         let left = b.hittable(&self.left)?;
///         let right = if Arc::ptr_eq(&self.left, &self.right) { left } else { b.hittable(&self.right)? };
///         b.nodes[i] = gpu::vk_node { bb_min: gpu::v3(self.bb.min), left, bb_max: gpu::v3(self.bb.max), right };
///         Ok(gpu::vk_mkref(gpu::VK_T_NODE, i as u32))
///     }
/// }
/// // The complete set -- every Hittable, Material and Texture the reference ships, Camera::lower, the call in main() --
/// // is rust/lower_impls.rs, block by block under the file each block is pasted into.  In short:
/// // FlipFace(Rect) sets VK_RECT_FLIP on a copy of the rect record; FlipFace of anything else,
/// // Translate and RotateX/Y/Z push one vk_xform {kind, child, a, b, c} (offset | sin, cos);
/// // Boxy pushes one vk_box; ConstantMedium one vk_medium {boundary.lower()?, -1/density, phase};
/// // Material::lower / Texture::lower push the tagged 16-byte records of vecchio_gpu.h.
/// ```
pub trait LowerDoc {}

impl Lowering {
    pub fn desc(&self, root: vk_ref) -> vk_scene_desc {
        vk_scene_desc {
            api_version: VK_API_VERSION, root,
            nodes: self.nodes.as_ptr(), n_nodes: self.nodes.len() as u32,
            spheres: self.spheres.as_ptr(), sphere_mat: self.sphere_mat.as_ptr(), n_spheres: self.spheres.len() as u32,
            mspheres: self.mspheres.as_ptr(), n_mspheres: self.mspheres.len() as u32,
            rects: self.rects.as_ptr(), n_rects: self.rects.len() as u32,
            boxes: self.boxes.as_ptr(), n_boxes: self.boxes.len() as u32,
            xforms: self.xforms.as_ptr(), n_xforms: self.xforms.len() as u32,
            media: self.media.as_ptr(), n_media: self.media.len() as u32,
            lights: self.lights.as_ptr(), n_lights: self.lights.len() as u32,
            materials: self.materials.as_ptr(), n_materials: self.materials.len() as u32,
            textures: self.textures.as_ptr(), n_textures: self.textures.len() as u32,
            texels: self.texels.as_ptr(), n_texel_bytes: self.texels.len() as u64,
            perlins: self.perlins.as_ptr(), n_perlins: self.perlins.len() as u32,
        }
    }
}

/// One GPU context; owns the device scene between frames (the 671-frame turntable of
/// random_spheres_demo uploads once and renders per camera).
pub struct Gpu { ctx: *mut vk_ctx }

impl Gpu {
    pub fn new(device: i32) -> Result<Gpu, GpuError> {
        let mut ctx = std::ptr::null_mut();
        let rc = unsafe { vk_create(device, &mut ctx) };
        if rc != 0 { return Err(GpuError::Library(rc, last_error(std::ptr::null()))); }
        Ok(Gpu { ctx })
    }
    fn check(&self, rc: c_int) -> Result<(), GpuError> {
        if rc == 0 { Ok(()) } else { Err(GpuError::Library(rc, last_error(self.ctx))) }
    }
    /// `world` is `Arc<BVHNode>` of src/main.rs:168, `lights` the Vec of :169 -- via their `lower()`.
    pub fn upload(&mut self, low: &Lowering, root: vk_ref) -> Result<(), GpuError> {
        let d = low.desc(root);
        self.check(unsafe { vk_scene_upload(self.ctx, &d) })
    }
    /// Replaces the body of src/main.rs:181-198.  Returns W*H*3 floats, pixel i = y*W + x, row 0 =
    /// bottom, linear mean over `spp` -- the layout of `pixels: Vec<Vec3>`.
    pub fn render(&mut self, cam: &vk_camera, width: usize, height: usize, spp: u32, max_depth: u32, seed: u64)
                  -> Result<(Vec<f32>, vk_stats), GpuError> {
        let p = vk_render_params { width: width as u32, height: height as u32, spp, spp_begin: 0, spp_count: 0, max_depth, seed,
                                   background: [0.0; 3], variant: 0, flags: 0 };
        let mut out = vec![0f32; width * height * 3];
        let mut st = vk_stats::default();
        self.check(unsafe { vk_render(self.ctx, cam, &p, out.as_mut_ptr(), std::ptr::null_mut(), &mut st) })?;
        Ok((out, st))
    }
    /// The same loop followed by `Vec3::to_color` and the top-down row order of src/main.rs:209-212 on the
    /// device: the W*H*3 numbers of the P3 file in file order (a quarter of the bytes cross PCIe).
    pub fn render_rgb8(&mut self, cam: &vk_camera, width: usize, height: usize, spp: u32, max_depth: u32, seed: u64)
                       -> Result<(Vec<u8>, vk_stats), GpuError> {
        let p = vk_render_params { width: width as u32, height: height as u32, spp, spp_begin: 0, spp_count: 0, max_depth, seed,
                                   background: [0.0; 3], variant: 0, flags: 0 };
        let mut out = vec![0u8; width * height * 3];
        let mut st = vk_stats::default();
        self.check(unsafe { vk_render_rgb8(self.ctx, cam, &p, out.as_mut_ptr(), &mut st) })?;
        Ok((out, st))
    }
    /// Several cameras of the turntable (`config.cam_iter`, src/main.rs:176) in one launch: frame f is
    /// `render_rgb8(&cams[f], .., seed + f)`, at offset f * W*H*3 of the result -- byte for byte when both run the same
    /// kernel; AUTO decides on the batch's path count, so a large batch may run a faster kernel, whose rounding differs
    /// in this (render) build.  The frames share the
    /// GPU's warps, so small frames fill it and the batch drains once.
    pub fn render_frames_rgb8(&mut self, cams: &[vk_camera], width: usize, height: usize, spp: u32, max_depth: u32, seed: u64)
                              -> Result<(Vec<u8>, vk_stats), GpuError> {
        if cams.is_empty() { return Err(GpuError::Unsupported("render_frames_rgb8: at least one camera")); }
        let p = vk_render_params { width: width as u32, height: height as u32, spp, spp_begin: 0, spp_count: 0, max_depth, seed,
                                   background: [0.0; 3], variant: 0, flags: 0 };
        let mut out = vec![0u8; cams.len() * width * height * 3];
        let mut st = vk_stats::default();
        self.check(unsafe { vk_render_frames_rgb8(self.ctx, cams.as_ptr(), cams.len() as u32, &p, out.as_mut_ptr(), &mut st) })?;
        Ok((out, st))
    }
    /// Feature buffers of K cameras for a denoiser (vk_render_aov in vecchio_gpu.h): first-hit albedo and normal (3 floats
    /// per pixel), depth and coverage (1 float), each frame in `render`'s layout, from the camera rays of samples
    /// 0 .. aov_spp-1 that `render_frames(.., seed, ..)` traces first.  Returns (albedo, normal, depth, coverage, stats).
    pub fn render_aov(&mut self, cams: &[vk_camera], width: usize, height: usize, seed: u64, aov_spp: u32)
                      -> Result<(Vec<f32>, Vec<f32>, Vec<f32>, Vec<f32>, vk_stats), GpuError> {
        if cams.is_empty() { return Err(GpuError::Unsupported("render_aov: at least one camera")); }
        let p = vk_render_params { width: width as u32, height: height as u32, spp: 1, spp_begin: 0, spp_count: 0, max_depth: 1, seed,
                                   background: [0.0; 3], variant: 0, flags: 0 };
        let n = cams.len() * width * height;
        let (mut albedo, mut normal, mut depth, mut coverage) = (vec![0f32; n * 3], vec![0f32; n * 3], vec![0f32; n], vec![0f32; n]);
        let mut st = vk_stats::default();
        self.check(unsafe { vk_render_aov(self.ctx, cams.as_ptr(), cams.len() as u32, &p, aov_spp, albedo.as_mut_ptr(), normal.as_mut_ptr(),
                                          depth.as_mut_ptr(), coverage.as_mut_ptr(), &mut st) })?;
        Ok((albedo, normal, depth, coverage, st))
    }
    /// Adaptive sampling with `spp` as the cap: every pixel renders passes of `pass_spp` samples until half the width of
    /// sqrt(mean +- standard error) is <= `max_error` 8-bit steps in every channel (vk_render_adaptive in vecchio_gpu.h).
    /// Returns the linear means in `render`'s layout and each pixel's sample count in the same order.  A pixel that
    /// stopped at n samples is `render(.., spp = n, ..)`'s pixel; the stopping rule makes the frame slightly biased.
    pub fn render_adaptive(&mut self, cam: &vk_camera, width: usize, height: usize, spp: u32, max_depth: u32, seed: u64,
                           pass_spp: u32, max_error: f32) -> Result<(Vec<f32>, Vec<u32>, vk_stats), GpuError> {
        let p = vk_render_params { width: width as u32, height: height as u32, spp, spp_begin: 0, spp_count: 0, max_depth, seed,
                                   background: [0.0; 3], variant: 0, flags: 0 };
        let mut out = vec![0f32; width * height * 3];
        let mut n = vec![0u32; width * height];
        let mut st = vk_stats::default();
        self.check(unsafe { vk_render_adaptive(self.ctx, cam, &p, pass_spp, max_error, out.as_mut_ptr(), n.as_mut_ptr(), &mut st) })?;
        Ok((out, n, st))
    }
    /// `render_adaptive` as `render_rgb8` returns a frame: the P3 file's numbers, the counts top-down as well.
    pub fn render_adaptive_rgb8(&mut self, cam: &vk_camera, width: usize, height: usize, spp: u32, max_depth: u32, seed: u64,
                                pass_spp: u32, max_error: f32) -> Result<(Vec<u8>, Vec<u32>, vk_stats), GpuError> {
        let p = vk_render_params { width: width as u32, height: height as u32, spp, spp_begin: 0, spp_count: 0, max_depth, seed,
                                   background: [0.0; 3], variant: 0, flags: 0 };
        let mut out = vec![0u8; width * height * 3];
        let mut n = vec![0u32; width * height];
        let mut st = vk_stats::default();
        self.check(unsafe { vk_render_adaptive_rgb8(self.ctx, cam, &p, pass_spp, max_error, out.as_mut_ptr(), n.as_mut_ptr(), &mut st) })?;
        Ok((out, n, st))
    }
    /// `render_adaptive` of K cameras, every pass one launch over the active pixels of all frames: frame f is
    /// `render_adaptive(&cams[f], .., seed + f, ..)`, at offset f * W*H*3 of the means and f * W*H of the counts -- bit for
    /// bit in the strict build; this (render) build may round some pixels differently (AUTO decides on the batch's pass-0 path count).
    pub fn render_frames_adaptive(&mut self, cams: &[vk_camera], width: usize, height: usize, spp: u32, max_depth: u32, seed: u64,
                                  pass_spp: u32, max_error: f32) -> Result<(Vec<f32>, Vec<u32>, vk_stats), GpuError> {
        if cams.is_empty() { return Err(GpuError::Unsupported("render_frames_adaptive: at least one camera")); }
        let p = vk_render_params { width: width as u32, height: height as u32, spp, spp_begin: 0, spp_count: 0, max_depth, seed,
                                   background: [0.0; 3], variant: 0, flags: 0 };
        let mut out = vec![0f32; cams.len() * width * height * 3];
        let mut n = vec![0u32; cams.len() * width * height];
        let mut st = vk_stats::default();
        self.check(unsafe { vk_render_frames_adaptive(self.ctx, cams.as_ptr(), cams.len() as u32, &p, pass_spp, max_error,
                                                      out.as_mut_ptr(), n.as_mut_ptr(), &mut st) })?;
        Ok((out, n, st))
    }
    /// `render_frames_adaptive` with every frame as `render_adaptive_rgb8` returns it (image and counts top-down).
    pub fn render_frames_adaptive_rgb8(&mut self, cams: &[vk_camera], width: usize, height: usize, spp: u32, max_depth: u32, seed: u64,
                                       pass_spp: u32, max_error: f32) -> Result<(Vec<u8>, Vec<u32>, vk_stats), GpuError> {
        if cams.is_empty() { return Err(GpuError::Unsupported("render_frames_adaptive_rgb8: at least one camera")); }
        let p = vk_render_params { width: width as u32, height: height as u32, spp, spp_begin: 0, spp_count: 0, max_depth, seed,
                                   background: [0.0; 3], variant: 0, flags: 0 };
        let mut out = vec![0u8; cams.len() * width * height * 3];
        let mut n = vec![0u32; cams.len() * width * height];
        let mut st = vk_stats::default();
        self.check(unsafe { vk_render_frames_adaptive_rgb8(self.ctx, cams.as_ptr(), cams.len() as u32, &p, pass_spp, max_error,
                                                           out.as_mut_ptr(), n.as_mut_ptr(), &mut st) })?;
        Ok((out, n, st))
    }
    /// One spp slice [begin, begin+count) of the frame, already divided by the full `spp`: slices of disjoint
    /// sample ranges ADD to the frame (the Philox counter holds the global sample index).
    pub fn render_slice(&mut self, cam: &vk_camera, width: usize, height: usize, spp: u32, begin: u32, count: u32,
                        max_depth: u32, seed: u64) -> Result<(Vec<f32>, vk_stats), GpuError> {
        let p = vk_render_params { width: width as u32, height: height as u32, spp, spp_begin: begin, spp_count: count, max_depth, seed,
                                   background: [0.0; 3], variant: 0, flags: 0 };
        let mut out = vec![0f32; width * height * 3];
        let mut st = vk_stats::default();
        self.check(unsafe { vk_render(self.ctx, cam, &p, out.as_mut_ptr(), std::ptr::null_mut(), &mut st) })?;
        Ok((out, st))
    }
    /// An adaptive render whose state outlives a call (vk_adaptive_begin): `refine` tightens it step by step, each step
    /// bit for bit a one-shot render at that target; `export` / `import` checkpoint it.  `spp` is the session's limit.
    /// The session borrows the context, so it cannot outlive it.
    pub fn adaptive_session(&mut self, cams: &[vk_camera], width: usize, height: usize, spp: u32, max_depth: u32, seed: u64,
                            pass_spp: u32) -> Result<AdaptiveSession<'_>, GpuError> {
        if cams.is_empty() { return Err(GpuError::Unsupported("adaptive_session: at least one camera")); }
        let p = vk_render_params { width: width as u32, height: height as u32, spp, spp_begin: 0, spp_count: 0, max_depth, seed,
                                   background: [0.0; 3], variant: 0, flags: 0 };
        let mut s = std::ptr::null_mut();
        self.check(unsafe { vk_adaptive_begin(self.ctx, cams.as_ptr(), cams.len() as u32, &p, pass_spp, &mut s) })?;
        Ok(AdaptiveSession { gpu: self, s, n_pix: cams.len() * width * height })
    }
}
impl Drop for Gpu { fn drop(&mut self) { unsafe { vk_destroy(self.ctx) } } }

/// A session of `Gpu::adaptive_session`; the lifetime ties it to its context.
pub struct AdaptiveSession<'a> { gpu: &'a mut Gpu, s: *mut vk_adaptive_session, n_pix: usize }
impl<'a> AdaptiveSession<'a> {
    /// Renders until `target` is reached; an error (and an unchanged state) for one that does not tighten the last.
    pub fn refine(&mut self, target: &vk_adaptive_target) -> Result<vk_stats, GpuError> {
        let mut st = vk_stats::default();
        self.gpu.check(unsafe { vk_adaptive_refine(self.s, target, &mut st) })?;
        Ok(st)
    }
    /// Means (rows bottom-up), counts and each pixel's error as the rule sees it (+inf below two samples).
    pub fn read(&mut self) -> Result<(Vec<f32>, Vec<u32>, Vec<f32>), GpuError> {
        let (mut out, mut n, mut e) = (vec![0f32; self.n_pix * 3], vec![0u32; self.n_pix], vec![0f32; self.n_pix]);
        self.gpu.check(unsafe { vk_adaptive_read(self.s, out.as_mut_ptr(), n.as_mut_ptr(), e.as_mut_ptr()) })?;
        Ok((out, n, e))
    }
    /// `read` as the P3 file holds the image: to_color, rows top-down, counts and errors in the same order.
    pub fn read_rgb8(&mut self) -> Result<(Vec<u8>, Vec<u32>, Vec<f32>), GpuError> {
        let (mut out, mut n, mut e) = (vec![0u8; self.n_pix * 3], vec![0u32; self.n_pix], vec![0f32; self.n_pix]);
        self.gpu.check(unsafe { vk_adaptive_read_rgb8(self.s, out.as_mut_ptr(), n.as_mut_ptr(), e.as_mut_ptr()) })?;
        Ok((out, n, e))
    }
    /// The raw state: fixed-point sums and squares (3 per pixel), counts, and the target reached.
    pub fn export(&mut self) -> Result<(Vec<i64>, Vec<u64>, Vec<u32>, vk_adaptive_target), GpuError> {
        let (mut sums, mut sq, mut n) = (vec![0i64; self.n_pix * 3], vec![0u64; self.n_pix * 3], vec![0u32; self.n_pix]);
        let mut t = vk_adaptive_target::default();
        self.gpu.check(unsafe { vk_adaptive_export(self.s, sums.as_mut_ptr(), sq.as_mut_ptr(), n.as_mut_ptr(), &mut t) })?;
        Ok((sums, sq, n, t))
    }
    /// Replaces the state by an exported one of a session with the same scene, cameras, params and pass_spp.
    pub fn import(&mut self, sums: &[i64], squares: &[u64], counts: &[u32], reached: &vk_adaptive_target) -> Result<(), GpuError> {
        if sums.len() != self.n_pix * 3 || squares.len() != self.n_pix * 3 || counts.len() != self.n_pix {
            return Err(GpuError::Unsupported("AdaptiveSession::import: array lengths do not match the session"));
        }
        self.gpu.check(unsafe { vk_adaptive_import(self.s, sums.as_ptr(), squares.as_ptr(), counts.as_ptr(), reached) })
    }
}
impl<'a> Drop for AdaptiveSession<'a> { fn drop(&mut self) { unsafe { vk_adaptive_destroy(self.s) } } }
// A context is used by one thread at a time and owns its device: it may move between threads.
unsafe impl Send for Gpu {}

/// Several GPUs in the reference's single process (what `vecchio_gpu_render --gpus N` does in C++,
/// vecchio_b200/host/main.cpp): ONE multi-device context.  Device k renders the global samples [k*spp/N, (k+1)*spp/N)
/// into its own integer accumulators; devices[0] adds its peers' accumulators over NVLink (peer-mapped memory) and
/// returns the frame -- bit-identical to the one-GPU frame for the same seed.
pub struct MultiGpu { m: *mut vk_multi }
impl MultiGpu {
    pub fn new(devices: &[i32]) -> Result<MultiGpu, GpuError> {
        let mut m = std::ptr::null_mut();
        let rc = unsafe { vk_multi_create(devices.as_ptr(), devices.len() as c_int, &mut m) };
        if rc != 0 { return Err(GpuError::Library(rc, multi_error(std::ptr::null()))); }
        Ok(MultiGpu { m })
    }
    fn check(&self, rc: c_int) -> Result<(), GpuError> {
        if rc == 0 { Ok(()) } else { Err(GpuError::Library(rc, multi_error(self.m))) }
    }
    pub fn upload(&mut self, low: &Lowering, root: vk_ref) -> Result<(), GpuError> {
        let d = low.desc(root);
        self.check(unsafe { vk_multi_scene_upload(self.m, &d) })
    }
    pub fn render(&mut self, cam: &vk_camera, width: usize, height: usize, spp: u32, max_depth: u32, seed: u64)
                  -> Result<(Vec<f32>, vk_stats), GpuError> {
        let p = vk_render_params { width: width as u32, height: height as u32, spp, spp_begin: 0, spp_count: 0, max_depth, seed,
                                   background: [0.0; 3], variant: 0, flags: 0 };
        let mut out = vec![0f32; width * height * 3];
        let mut st = vk_stats::default();
        self.check(unsafe { vk_multi_render(self.m, cam, &p, out.as_mut_ptr(), std::ptr::null_mut(), &mut st) })?;
        Ok((out, st))
    }
    /// `Gpu::render_frames_rgb8` over all devices (every device renders its sample slice of every frame): the same bytes as one GPU's batch.
    pub fn render_frames_rgb8(&mut self, cams: &[vk_camera], width: usize, height: usize, spp: u32, max_depth: u32, seed: u64)
                              -> Result<(Vec<u8>, vk_stats), GpuError> {
        if cams.is_empty() { return Err(GpuError::Unsupported("render_frames_rgb8: at least one camera")); }
        let p = vk_render_params { width: width as u32, height: height as u32, spp, spp_begin: 0, spp_count: 0, max_depth, seed,
                                   background: [0.0; 3], variant: 0, flags: 0 };
        let mut out = vec![0u8; cams.len() * width * height * 3];
        let mut st = vk_stats::default();
        self.check(unsafe { vk_multi_render_frames_rgb8(self.m, cams.as_ptr(), cams.len() as u32, &p, out.as_mut_ptr(), &mut st) })?;
        Ok((out, st))
    }
    /// `Gpu::render_adaptive_rgb8` over all devices (device k renders the pixels of shard k): the same bytes and counts.
    pub fn render_adaptive_rgb8(&mut self, cam: &vk_camera, width: usize, height: usize, spp: u32, max_depth: u32, seed: u64,
                                pass_spp: u32, max_error: f32) -> Result<(Vec<u8>, Vec<u32>, vk_stats), GpuError> {
        let p = vk_render_params { width: width as u32, height: height as u32, spp, spp_begin: 0, spp_count: 0, max_depth, seed,
                                   background: [0.0; 3], variant: 0, flags: 0 };
        let mut out = vec![0u8; width * height * 3];
        let mut n = vec![0u32; width * height];
        let mut st = vk_stats::default();
        self.check(unsafe { vk_multi_render_adaptive_rgb8(self.m, cam, &p, pass_spp, max_error, out.as_mut_ptr(), n.as_mut_ptr(), &mut st) })?;
        Ok((out, n, st))
    }
    /// `Gpu::render_frames_adaptive_rgb8` over all devices: the same bytes and counts as one GPU's batch.
    pub fn render_frames_adaptive_rgb8(&mut self, cams: &[vk_camera], width: usize, height: usize, spp: u32, max_depth: u32, seed: u64,
                                       pass_spp: u32, max_error: f32) -> Result<(Vec<u8>, Vec<u32>, vk_stats), GpuError> {
        if cams.is_empty() { return Err(GpuError::Unsupported("render_frames_adaptive_rgb8: at least one camera")); }
        let p = vk_render_params { width: width as u32, height: height as u32, spp, spp_begin: 0, spp_count: 0, max_depth, seed,
                                   background: [0.0; 3], variant: 0, flags: 0 };
        let mut out = vec![0u8; cams.len() * width * height * 3];
        let mut n = vec![0u32; cams.len() * width * height];
        let mut st = vk_stats::default();
        self.check(unsafe { vk_multi_render_frames_adaptive_rgb8(self.m, cams.as_ptr(), cams.len() as u32, &p, pass_spp, max_error,
                                                                 out.as_mut_ptr(), n.as_mut_ptr(), &mut st) })?;
        Ok((out, n, st))
    }
    /// `Gpu::adaptive_session` over all devices (vk_multi_adaptive_begin): the same results, and checkpoints that move
    /// between one GPU and several.  The session borrows the MultiGpu.
    pub fn adaptive_session(&mut self, cams: &[vk_camera], width: usize, height: usize, spp: u32, max_depth: u32, seed: u64,
                            pass_spp: u32) -> Result<MultiAdaptiveSession<'_>, GpuError> {
        if cams.is_empty() { return Err(GpuError::Unsupported("adaptive_session: at least one camera")); }
        let p = vk_render_params { width: width as u32, height: height as u32, spp, spp_begin: 0, spp_count: 0, max_depth, seed,
                                   background: [0.0; 3], variant: 0, flags: 0 };
        let mut s = std::ptr::null_mut();
        self.check(unsafe { vk_multi_adaptive_begin(self.m, cams.as_ptr(), cams.len() as u32, &p, pass_spp, &mut s) })?;
        Ok(MultiAdaptiveSession { multi: self, s, n_pix: cams.len() * width * height })
    }
}
impl Drop for MultiGpu { fn drop(&mut self) { unsafe { vk_multi_destroy(self.m) } } }

/// A session of `MultiGpu::adaptive_session`: `AdaptiveSession`'s methods over all devices.
pub struct MultiAdaptiveSession<'a> { multi: &'a mut MultiGpu, s: *mut vk_multi_adaptive_session, n_pix: usize }
impl<'a> MultiAdaptiveSession<'a> {
    pub fn refine(&mut self, target: &vk_adaptive_target) -> Result<vk_stats, GpuError> {
        let mut st = vk_stats::default();
        self.multi.check(unsafe { vk_multi_adaptive_refine(self.s, target, &mut st) })?;
        Ok(st)
    }
    pub fn read(&mut self) -> Result<(Vec<f32>, Vec<u32>, Vec<f32>), GpuError> {
        let (mut out, mut n, mut e) = (vec![0f32; self.n_pix * 3], vec![0u32; self.n_pix], vec![0f32; self.n_pix]);
        self.multi.check(unsafe { vk_multi_adaptive_read(self.s, out.as_mut_ptr(), n.as_mut_ptr(), e.as_mut_ptr()) })?;
        Ok((out, n, e))
    }
    pub fn read_rgb8(&mut self) -> Result<(Vec<u8>, Vec<u32>, Vec<f32>), GpuError> {
        let (mut out, mut n, mut e) = (vec![0u8; self.n_pix * 3], vec![0u32; self.n_pix], vec![0f32; self.n_pix]);
        self.multi.check(unsafe { vk_multi_adaptive_read_rgb8(self.s, out.as_mut_ptr(), n.as_mut_ptr(), e.as_mut_ptr()) })?;
        Ok((out, n, e))
    }
    pub fn export(&mut self) -> Result<(Vec<i64>, Vec<u64>, Vec<u32>, vk_adaptive_target), GpuError> {
        let (mut sums, mut sq, mut n) = (vec![0i64; self.n_pix * 3], vec![0u64; self.n_pix * 3], vec![0u32; self.n_pix]);
        let mut t = vk_adaptive_target::default();
        self.multi.check(unsafe { vk_multi_adaptive_export(self.s, sums.as_mut_ptr(), sq.as_mut_ptr(), n.as_mut_ptr(), &mut t) })?;
        Ok((sums, sq, n, t))
    }
    pub fn import(&mut self, sums: &[i64], squares: &[u64], counts: &[u32], reached: &vk_adaptive_target) -> Result<(), GpuError> {
        if sums.len() != self.n_pix * 3 || squares.len() != self.n_pix * 3 || counts.len() != self.n_pix {
            return Err(GpuError::Unsupported("MultiAdaptiveSession::import: array lengths do not match the session"));
        }
        self.multi.check(unsafe { vk_multi_adaptive_import(self.s, sums.as_ptr(), squares.as_ptr(), counts.as_ptr(), reached) })
    }
}
impl<'a> Drop for MultiAdaptiveSession<'a> { fn drop(&mut self) { unsafe { vk_multi_adaptive_destroy(self.s) } } }
unsafe impl Send for MultiGpu {}
fn multi_error(m: *const vk_multi) -> String {
    unsafe { let p = vk_multi_last_error(m); if p.is_null() { String::new() } else { CStr::from_ptr(p).to_string_lossy().into_owned() } }
}

fn last_error(ctx: *const vk_ctx) -> String {
    unsafe { let p = vk_last_error(ctx); if p.is_null() { String::new() } else { CStr::from_ptr(p).to_string_lossy().into_owned() } }
}

// Camera -> vk_camera: the ten fields of src/main.rs:56-68 in declaration order (a `lower()` on
// Camera inside main.rs, because its fields are private):
//   vk_camera { origin: self.origin.into(), lower_left_corner: .., horizontal: .., vertical: ..,
//               u: .., v: .., w: .., lens_radius: self.lens_radius, time0: self.time0, time1: self.time1 }
