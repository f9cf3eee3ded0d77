//! gpu_ffi.rs — binding of librtb200.so for the ray-tracing-series-rust crate (SOURCE ONLY: this image has no Rust
//! toolchain, so the file has never been compiled; the same call sequence is exercised from C++ in
//! ray_tracing_series_rust_b200/csrc/host/world.hpp and from Python in ray_tracing_series_rust_b200/capi.py).
//!
//! How to apply it to the reference crate:
//!   1. copy this file to src/gpu_ffi.rs and add `pub mod gpu_ffi;` to src/lib.rs;
//!   2. make the struct fields it reads `pub(crate)` (hit.rs, texture.rs, perlin.rs, camera.rs, bvh.rs, screen.rs) — they are
//!      private today and the traits cannot be downcast, which is why the shim has to live inside the crate;
//!   3. add the flatten traits below as supertraits:  `pub trait Hittable: FlattenHittable + Send + Sync`,
//!      `pub trait Material: FlattenMaterial`, `pub trait Texture: FlattenTexture`   (hit.rs:82, hit.rs:1013, texture.rs:7);
//!   4. link: `println!("cargo:rustc-link-lib=dylib=rtb200");` in build.rs (+ rustc-link-search to the directory of the .so);
//!   5. call `render_scene_gpu` where main.rs:10-13 calls `render_scene`.
//!
//! Every `rt_*` call mirrors one reference constructor; ids mirror `Arc` sharing (one id per Arc allocation).
use std::collections::HashMap;
use std::ffi::{CStr, CString};
use std::os::raw::c_char;
use std::sync::Arc;

use crate::bvh::BvhNode;
use crate::camera::Camera;
use crate::hit::*;
use crate::screen::Screen;
use crate::texture::*;
use crate::vec3::{Color, Vec3};
use crate::world::Config;

#[repr(C)]
pub struct RtScene {
    _private: [u8; 0],
}

/// rt_render_config (include/rtb200.h) <-> Config (src/world.rs:20-26)
#[repr(C)]
pub struct RtRenderConfig {
    pub image_width: i32,
    pub aspect_ratio: f64,
    pub samples_per_pixel: i32,
    pub max_depth: i32,
    pub compat_threads: i32, // Config.threads: reproduces the H - N*(H/N) unrendered rows (world.rs:1198-1202); 0 = all rows
    pub seed: u64,
    pub sample_begin: i32,
    pub sample_end: i32,
    pub threads: i32,
    pub flags: i32,
}

/// rt_adaptive_config (include/rtb200.h): per-pixel sample counts for rt_render_adaptive
#[repr(C)]
pub struct RtAdaptiveConfig {
    pub min_samples: i32, // 0 ..= samples_per_pixel: no pixel stops before this many samples
    pub step: i32,        // >= 1: samples per round; check points every 2 rounds
    pub threshold: f64,   // >= 0 and finite; 0 = no pixel converges (result == rt_render)
    pub radius: i32,      // 0..=8: a pixel stays active while an unconverged pixel is this close
}

#[link(name = "rtb200")]
extern "C" {
    fn rt_scene_create() -> *mut RtScene;
    fn rt_scene_destroy(s: *mut RtScene);
    fn rt_last_error() -> *const c_char;
    fn rt_tex_solid(s: *mut RtScene, rgb: *const f64) -> i32;
    fn rt_tex_checker(s: *mut RtScene, even: i32, odd: i32) -> i32;
    fn rt_tex_noise(s: *mut RtScene, scale: f64, ranvec: *const f64, px: *const i32, py: *const i32, pz: *const i32, seed: u64) -> i32;
    fn rt_tex_image(s: *mut RtScene, w: i32, h: i32, rgb: *const f64) -> i32;
    fn rt_mat_lambertian(s: *mut RtScene, tex: i32) -> i32;
    fn rt_mat_metal(s: *mut RtScene, albedo: *const f64, fuzz: f64) -> i32;
    fn rt_mat_dielectric(s: *mut RtScene, ir: f64) -> i32;
    fn rt_mat_diffuse_light(s: *mut RtScene, tex: i32) -> i32;
    fn rt_mat_isotropic(s: *mut RtScene, tex: i32) -> i32;
    fn rt_sphere(s: *mut RtScene, c: *const f64, r: f64, mat: i32) -> i32;
    fn rt_moving_sphere(s: *mut RtScene, c0: *const f64, c1: *const f64, t0: f64, t1: f64, r: f64, mat: i32) -> i32;
    fn rt_gravity_sphere(s: *mut RtScene, start: *const f64, time0: f64, r: f64, mat: i32) -> i32;
    fn rt_xy_rect(s: *mut RtScene, x0: f64, x1: f64, y0: f64, y1: f64, k: f64, mat: i32) -> i32;
    fn rt_xz_rect(s: *mut RtScene, x0: f64, x1: f64, z0: f64, z1: f64, k: f64, mat: i32) -> i32;
    fn rt_yz_rect(s: *mut RtScene, y0: f64, y1: f64, z0: f64, z1: f64, k: f64, mat: i32) -> i32;
    fn rt_box(s: *mut RtScene, p0: *const f64, p1: *const f64, mat: i32) -> i32;
    fn rt_triangle(s: *mut RtScene, v0: *const f64, v1: *const f64, v2: *const f64, mat: i32) -> i32;
    fn rt_list(s: *mut RtScene, ids: *const i32, n: i32) -> i32;
    fn rt_bvh(s: *mut RtScene, ids: *const i32, n: i32, t0: f64, t1: f64) -> i32;
    fn rt_translate(s: *mut RtScene, off: *const f64, child: i32) -> i32;
    fn rt_rotate_y(s: *mut RtScene, angle_deg: f64, child: i32) -> i32;
    fn rt_constant_medium(s: *mut RtScene, rgb: *const f64, density: f64, boundary: i32) -> i32;
    fn rt_scene_set_root(s: *mut RtScene, id: i32) -> i32;
    fn rt_scene_set_camera_fields(s: *mut RtScene, fields: *const f64) -> i32;
    fn rt_scene_set_background(s: *mut RtScene, rgb: *const f64) -> i32;
    fn rt_scene_set_background_gradient(s: *mut RtScene, horizon_rgb: *const f64, zenith_rgb: *const f64) -> i32;
    fn rt_scene_commit(s: *mut RtScene) -> i32;
    fn rt_scene_commit_multi(s: *mut RtScene, n_gpus: i32) -> i32;
    fn rt_image_height(cfg: *const RtRenderConfig) -> i32;
    fn rt_render(s: *mut RtScene, cfg: *const RtRenderConfig, out_screen: *mut f64, out_accum: *mut i64, stats: *mut u8) -> i32;
    /// one host thread, n_gpus devices of the box: shards rendered per GPU, summed + resolved over NVLink peer memory (include/rtb200.h)
    fn rt_render_multi(s: *mut RtScene, cfg: *const RtRenderConfig, n_gpus: i32, shard_mode: i32, out_screen: *mut f64, out_accum: *mut i64, stats: *mut u8) -> i32;
    /// every pixel until its noise estimate converges, at most cfg.samples_per_pixel; out_samples = W*H per-pixel counts (nullable)
    fn rt_render_adaptive(s: *mut RtScene, cfg: *const RtRenderConfig, ac: *const RtAdaptiveConfig, out_screen: *mut f64, out_accum: *mut i64,
                          out_samples: *mut i32, stats: *mut u8) -> i32;
    /// rt_render_adaptive with every round's paths spread over n_gpus devices of the box; bit-identical to it for every n_gpus
    fn rt_render_adaptive_multi(s: *mut RtScene, cfg: *const RtRenderConfig, ac: *const RtAdaptiveConfig, n_gpus: i32, out_screen: *mut f64,
                                out_accum: *mut i64, out_samples: *mut i32, stats: *mut u8) -> i32;
    fn rt_render_scene_with_time(s: *mut RtScene, t0: f64, t1: f64, path: *const c_char, cfg: *const RtRenderConfig, out_screen: *mut f64, stats: *mut u8) -> i32;
    fn rt_write_ppm(path: *const c_char, screen: *const f64, w: i32, h: i32) -> i32;
}

pub const RT_SHARD_SAMPLES: i32 = 0; // contiguous sample ranges of every pixel per GPU (perfect balance)
pub const RT_SHARD_TILES: i32 = 1; // 4-row bands dealt round-robin (the reference's row bands, world.rs:1198-1227)

/// GPUs to use: RTB200_GPUS in the environment, else 1 (the library refuses more than the box has).
fn n_gpus() -> i32 {
    std::env::var("RTB200_GPUS").ok().and_then(|v| v.parse().ok()).unwrap_or(1)
}

/// The reference panics where the C-ABI returns a negative rt_status (world.rs:36-40, screen.rs:14, bvh.rs:27-28, model.rs:15).
fn check(code: i32) -> i32 {
    if code < 0 {
        let msg = unsafe { CStr::from_ptr(rt_last_error()) }.to_string_lossy().into_owned();
        panic!("rtb200: rt_status {}: {}", code, msg);
    }
    code
}

fn xyz(v: &Vec3) -> [f64; 3] {
    [v.get_x(), v.get_y(), v.get_z()]
}

/// Builder handed down the scene graph.  `seen` memoises ids by Arc allocation so that a shared object is created once.
pub struct FlatSceneBuilder {
    pub s: *mut RtScene,
    seen: HashMap<usize, i32>,
}

impl FlatSceneBuilder {
    pub fn new() -> FlatSceneBuilder {
        FlatSceneBuilder { s: unsafe { rt_scene_create() }, seen: HashMap::new() }
    }
    fn memo<T: ?Sized>(&mut self, p: *const T, make: impl FnOnce(&mut FlatSceneBuilder) -> i32) -> i32 {
        let key = p as *const u8 as usize;
        if let Some(id) = self.seen.get(&key) {
            return *id;
        }
        let id = make(self);
        self.seen.insert(key, id);
        id
    }
    pub fn hittable(&mut self, o: &Arc<Box<dyn Hittable + Sync>>) -> i32 {
        self.memo(Arc::as_ptr(o), |b| o.flatten(b))
    }
    pub fn hittable_send(&mut self, o: &Arc<Box<dyn Hittable + Send + Sync>>) -> i32 {
        self.memo(Arc::as_ptr(o), |b| o.flatten(b))
    }
    pub fn hittable_plain(&mut self, o: &Arc<Box<dyn Hittable>>) -> i32 {
        self.memo(Arc::as_ptr(o), |b| o.flatten(b))
    }
    pub fn material(&mut self, m: &Arc<Box<dyn Material>>) -> i32 {
        self.memo(Arc::as_ptr(m), |b| m.flatten(b))
    }
    pub fn texture(&mut self, t: &Arc<Box<dyn Texture>>) -> i32 {
        self.memo(Arc::as_ptr(t), |b| t.flatten(b))
    }
}

impl Drop for FlatSceneBuilder {
    fn drop(&mut self) {
        unsafe { rt_scene_destroy(self.s) }
    }
}

pub trait FlattenHittable {
    fn flatten(&self, b: &mut FlatSceneBuilder) -> i32;
}
pub trait FlattenMaterial {
    fn flatten(&self, b: &mut FlatSceneBuilder) -> i32;
}
pub trait FlattenTexture {
    fn flatten(&self, b: &mut FlatSceneBuilder) -> i32;
}

// ------------------------------------------------------------------ textures (texture.rs)
impl FlattenTexture for SolidColor {
    fn flatten(&self, b: &mut FlatSceneBuilder) -> i32 {
        check(unsafe { rt_tex_solid(b.s, xyz(&self.color_value).as_ptr()) })
    }
}
impl FlattenTexture for Checker {
    fn flatten(&self, b: &mut FlatSceneBuilder) -> i32 {
        let (e, o) = (b.texture(&self.even), b.texture(&self.odd));
        check(unsafe { rt_tex_checker(b.s, e, o) })
    }
}
impl FlattenTexture for Noise {
    // the Perlin tables are DATA: passed exactly as Perlin::new drew them (perlin.rs:14-26, 68-83)
    fn flatten(&self, b: &mut FlatSceneBuilder) -> i32 {
        let rv: Vec<f64> = self.noise.ranvec.iter().flat_map(|v| xyz(v)).collect();
        check(unsafe {
            rt_tex_noise(b.s, self.scale, rv.as_ptr(), self.noise.perm_x.as_ptr(), self.noise.perm_y.as_ptr(), self.noise.perm_z.as_ptr(), 0)
        })
    }
}
impl FlattenTexture for Image {
    // Screen::from_ppm_p3 keeps the file's rows in file order (screen.rs:61-95) and Image::value indexes them with the flipped v
    // (texture.rs:102-121): row 0 = top of the file, which is what rt_tex_image expects
    fn flatten(&self, b: &mut FlatSceneBuilder) -> i32 {
        let (w, h) = (self.data.width, self.data.height);
        let mut rgb: Vec<f64> = Vec::with_capacity(w * h * 3);
        for j in 0..h {
            for i in 0..w {
                rgb.extend_from_slice(&xyz(self.data.get(j, i)));
            }
        }
        check(unsafe { rt_tex_image(b.s, w as i32, h as i32, rgb.as_ptr()) })
    }
}

// ------------------------------------------------------------------ materials (hit.rs:992-1152)
impl FlattenMaterial for Lambertian {
    fn flatten(&self, b: &mut FlatSceneBuilder) -> i32 {
        let t = b.texture(&self.albedo);
        check(unsafe { rt_mat_lambertian(b.s, t) })
    }
}
impl FlattenMaterial for Metal {
    fn flatten(&self, b: &mut FlatSceneBuilder) -> i32 {
        check(unsafe { rt_mat_metal(b.s, xyz(&self.albedo).as_ptr(), self.fuzz) })
    }
}
impl FlattenMaterial for Dielectric {
    fn flatten(&self, b: &mut FlatSceneBuilder) -> i32 {
        check(unsafe { rt_mat_dielectric(b.s, self.ir) })
    }
}
impl FlattenMaterial for DiffuseLight {
    fn flatten(&self, b: &mut FlatSceneBuilder) -> i32 {
        let t = b.texture(&self.emit);
        check(unsafe { rt_mat_diffuse_light(b.s, t) })
    }
}
impl FlattenMaterial for Isotropic {
    fn flatten(&self, b: &mut FlatSceneBuilder) -> i32 {
        let t = b.texture(&self.albedo);
        check(unsafe { rt_mat_isotropic(b.s, t) })
    }
}

// ------------------------------------------------------------------ hittables (hit.rs, bvh.rs)
impl FlattenHittable for Sphere {
    fn flatten(&self, b: &mut FlatSceneBuilder) -> i32 {
        let m = b.material(&self.mat_ptr);
        check(unsafe { rt_sphere(b.s, xyz(&self.center).as_ptr(), self.radius, m) })
    }
}
impl FlattenHittable for MovingSphere {
    fn flatten(&self, b: &mut FlatSceneBuilder) -> i32 {
        let m = b.material(&self.mat_ptr);
        check(unsafe { rt_moving_sphere(b.s, xyz(&self.center0).as_ptr(), xyz(&self.center1).as_ptr(), self.time0, self.time1, self.radius, m) })
    }
}
impl FlattenHittable for GravitySphere {
    // the library re-integrates the bounce table from (start, time0, radius) exactly as hit.rs:346-359 does
    fn flatten(&self, b: &mut FlatSceneBuilder) -> i32 {
        let m = b.material(&self.mat_ptr);
        check(unsafe { rt_gravity_sphere(b.s, xyz(&self.start).as_ptr(), self.time0, self.radius, m) })
    }
}
impl FlattenHittable for XyRect {
    fn flatten(&self, b: &mut FlatSceneBuilder) -> i32 {
        let m = b.material(&self.mat_ptr);
        check(unsafe { rt_xy_rect(b.s, self.x0, self.x1, self.y0, self.y1, self.k, m) })
    }
}
impl FlattenHittable for XzRect {
    // the reference names the fields x0,x1,y0,y1 in all three rects; here they are the (x, z) extents (hit.rs:511-519)
    fn flatten(&self, b: &mut FlatSceneBuilder) -> i32 {
        let m = b.material(&self.mat_ptr);
        check(unsafe { rt_xz_rect(b.s, self.x0, self.x1, self.y0, self.y1, self.k, m) })
    }
}
impl FlattenHittable for YzRect {
    fn flatten(&self, b: &mut FlatSceneBuilder) -> i32 {
        let m = b.material(&self.mat_ptr);
        check(unsafe { rt_yz_rect(b.s, self.x0, self.x1, self.y0, self.y1, self.k, m) })
    }
}
impl FlattenHittable for Triangle {
    fn flatten(&self, b: &mut FlatSceneBuilder) -> i32 {
        let m = b.material(&self.mat_ptr);
        check(unsafe { rt_triangle(b.s, xyz(&self.v0).as_ptr(), xyz(&self.v1).as_ptr(), xyz(&self.v2).as_ptr(), m) })
    }
}
impl FlattenHittable for RectPrism {
    // one primitive on the device; its six sides keep the ids and the scan order of hit.rs:722-769.
    // RectPrism::new hands one material to all six rects: take it from the first side.
    fn flatten(&self, b: &mut FlatSceneBuilder) -> i32 {
        let m = b.material(&self.mat);  // add `mat: Arc<Box<dyn Material>>` to RectPrism (it is consumed by `new` today)
        check(unsafe { rt_box(b.s, xyz(&self.box_min).as_ptr(), xyz(&self.box_max).as_ptr(), m) })
    }
}
impl FlattenHittable for HittableList {
    fn flatten(&self, b: &mut FlatSceneBuilder) -> i32 {
        let ids: Vec<i32> = self.objects.iter().map(|o| b.hittable(o)).collect();
        check(unsafe { rt_list(b.s, ids.as_ptr(), ids.len() as i32) })
    }
}
impl FlattenHittable for BvhNode {
    // The random median-split tree is not exported, its objects are: closest hit does not depend on topology
    // (bvh.rs:97-112).  A single-leaf node holds the same Arc twice (bvh.rs:53-55): pass it once.
    // The library bounds moving primitives over the camera shutter, so the (time0, time1) of from_list are not needed.
    fn flatten(&self, b: &mut FlatSceneBuilder) -> i32 {
        let l = b.hittable(&self.left);
        let ids = if Arc::ptr_eq(&self.left, &self.right) { vec![l] } else { vec![l, b.hittable(&self.right)] };
        check(unsafe { rt_bvh(b.s, ids.as_ptr(), ids.len() as i32, 0.0, 1.0) })
    }
}
impl FlattenHittable for Translate {
    fn flatten(&self, b: &mut FlatSceneBuilder) -> i32 {
        let c = b.hittable_send(&self.obj);
        check(unsafe { rt_translate(b.s, xyz(&self.offset).as_ptr(), c) })
    }
}
impl FlattenHittable for RotateY {
    // RotateY::new keeps sin/cos, not the angle (hit.rs:843-888): recover the degrees the constructor was given
    fn flatten(&self, b: &mut FlatSceneBuilder) -> i32 {
        let c = b.hittable_send(&self.obj);
        let deg = self.sin_theta.atan2(self.cos_theta).to_degrees();
        check(unsafe { rt_rotate_y(b.s, deg, c) })
    }
}
impl FlattenHittable for ConstantMedium {
    // phase_function is always Isotropic(SolidColor(c)) (hit.rs:945-951); the library creates it from (colour, density).
    // Keep `color: Color` and `density: f64` next to neg_inv_density, or read them back: density = -1 / neg_inv_density.
    fn flatten(&self, b: &mut FlatSceneBuilder) -> i32 {
        let bd = b.hittable_plain(&self.boundary);
        check(unsafe { rt_constant_medium(b.s, xyz(&self.color).as_ptr(), -1.0 / self.neg_inv_density, bd) })
    }
}

impl Camera {
    /// The 24 stored f64 of the struct (camera.rs:6-17) in declaration order.
    pub fn flatten(&self, b: &mut FlatSceneBuilder) {
        let mut f: Vec<f64> = Vec::with_capacity(24);
        for v in [&self.origin, &self.lower_left_corner, &self.horizontal, &self.vertical, &self.u, &self.v, &self.w] {
            f.extend_from_slice(&xyz(v));
        }
        f.extend_from_slice(&[self.lens_radius, self.time1, self.time2]);
        check(unsafe { rt_scene_set_camera_fields(b.s, f.as_ptr()) });
    }
}

/// Drop-in for `render_scene` (src/world.rs:1181-1247): same arguments, same P3 PPM on stdout.  With RTB200_GPUS=8 the same call
/// drives the whole 8 x B200 node (rt_render_multi): the image is bit-identical for every GPU count.
pub fn render_scene_gpu(world: Arc<Box<dyn Hittable + Sync>>, cam: Arc<Camera>, background: Vec3, config: Config) {
    let mut b = FlatSceneBuilder::new();
    let root = b.hittable(&world);
    check(unsafe { rt_scene_set_root(b.s, root) });
    cam.flatten(&mut b);
    check(unsafe { rt_scene_set_background(b.s, xyz(&background).as_ptr()) });
    let gpus = n_gpus();
    check(unsafe { rt_scene_commit_multi(b.s, gpus) }); // flatten + BVH build + one upload per GPU
    let cfg = RtRenderConfig {
        image_width: config.image_width,
        aspect_ratio: config.aspect_ratio,
        samples_per_pixel: config.samples_per_pixel,
        max_depth: config.max_depth,
        compat_threads: config.threads as i32,
        seed: 1,
        sample_begin: 0,
        sample_end: 0,
        threads: 0,
        flags: 0,
    };
    let h = check(unsafe { rt_image_height(&cfg) }) as usize;
    let w = config.image_width as usize;
    let mut pixels = vec![0.0f64; w * h * 3]; // Screen layout: row 0 = bottom, integer-valued 0..255 (vec3.rs:89-107)
    check(unsafe { rt_render_multi(b.s, &cfg, gpus, RT_SHARD_SAMPLES, pixels.as_mut_ptr(), std::ptr::null_mut(), std::ptr::null_mut()) });
    check(unsafe { rt_write_ppm(std::ptr::null(), pixels.as_ptr(), w as i32, h as i32) }); // byte-identical to Screen::write_to_ppm
}

/// Drop-in for `render_scene_with_time(t0, t1, path, world)` (src/world.rs:1249-1330): binds the library's own frame entry, which
/// sets the reference's hard-coded frame camera ((13,2,3) -> 0, vfov 20, aperture 0.1, focus 10, shutter [t0, t1)) and background,
/// re-commits (GravitySphere windows and moving bounds follow the shutter), renders and writes the P3 file.  `cfg` = None gives
/// the reference's 500 x 500, 500 spp, depth 50, 11 row bands.
pub fn render_frame_gpu(b: &mut FlatSceneBuilder, t0: f64, t1: f64, path: &str, cfg: Option<&RtRenderConfig>) -> Screen {
    let probe = RtRenderConfig { image_width: 500, aspect_ratio: 1.0, samples_per_pixel: 500, max_depth: 50, compat_threads: 11, seed: 1,
                                 sample_begin: 0, sample_end: 0, threads: 0, flags: 0 };
    let c: &RtRenderConfig = cfg.unwrap_or(&probe);
    let h = check(unsafe { rt_image_height(c) }) as usize;
    let w = c.image_width as usize;
    let mut pixels = vec![0.0f64; w * h * 3];
    let cpath = CString::new(path).unwrap();
    let cfg_ptr = match cfg { Some(p) => p as *const RtRenderConfig, None => std::ptr::null() };
    check(unsafe { rt_render_scene_with_time(b.s, t0, t1, cpath.as_ptr(), cfg_ptr, pixels.as_mut_ptr(), std::ptr::null_mut()) });
    let mut screen = Screen::new(w, h);
    for j in 0..h {
        for i in 0..w {
            let o = (j * w + i) * 3;
            screen.update(j, i, Color::new(pixels[o], pixels[o + 1], pixels[o + 2]));
        }
    }
    screen
}

/// The sky of the revision that rendered images/book1.png (README.md:18): not in HEAD's ray_color (world.rs:86-89 has the constant
/// background only); exposed so that renders can be checked against that shipped image.
pub fn set_book1_sky(b: &mut FlatSceneBuilder) {
    let (horizon, zenith) = ([1.0f64, 1.0, 1.0], [0.5f64, 0.7, 1.0]);
    check(unsafe { rt_scene_set_background_gradient(b.s, horizon.as_ptr(), zenith.as_ptr()) });
}
