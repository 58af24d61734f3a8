//! Safe wrapper over the C ABI (`include/shimmer_b200.h`).  One method per reference constructor; ids are plain
//! newtypes; every call maps `< 0` to `Error` with the library's message.  There is no CPU fallback: without a CUDA
//! device `commit`/`render` return `Error { code: SHIM_ERR_CUDA, .. }`.
//! NOTE: written without a Rust toolchain at hand (the build image has none), so this crate, `trace_hit` and
//! `trace_occluded` included, has never been compiled; see rust/README.md.
use std::ffi::{CStr, CString};
use std::ops::{Deref, DerefMut};
use std::os::raw::c_int;

pub use shimmer_b200_sys as sys;
pub use sys::{shim_camera as Camera, shim_render_params as RenderParams, shim_stats as Stats};

#[derive(Debug, Clone)]
pub struct Error {
    pub code: i32,
    pub message: String,
}
impl std::fmt::Display for Error {
    fn fmt(&self, f: &mut std::fmt::Formatter<'_>) -> std::fmt::Result {
        write!(f, "shimmer-b200 error {}: {}", self.code, self.message)
    }
}
impl std::error::Error for Error {}
impl From<Error> for std::io::Error {
    fn from(e: Error) -> Self {
        std::io::Error::new(std::io::ErrorKind::Other, e)
    }
}
pub type Result<T> = std::result::Result<T, Error>;

fn last_error(code: c_int) -> Error {
    let message = unsafe {
        let p = sys::shim_last_error();
        if p.is_null() { String::new() } else { CStr::from_ptr(p).to_string_lossy().into_owned() }
    };
    Error { code, message }
}
fn check(rc: c_int) -> Result<i32> {
    if rc < 0 { Err(last_error(rc)) } else { Ok(rc) }
}

#[derive(Clone, Copy, Debug, PartialEq, Eq, Hash)]
pub struct TextureId(pub i32);
#[derive(Clone, Copy, Debug, PartialEq, Eq, Hash)]
pub struct MaterialId(pub i32);
/// Also the primitive id `trace_closest` reports.
#[derive(Clone, Copy, Debug, PartialEq, Eq, Hash)]
pub struct HittableId(pub i32);

/// `HitRecord` (hittable.rs:15-52) as `Scene::trace_hit` returns it, with the id of the hittable that answered (the id
/// `trace_closest` reports; a ConstantMedium hit: the medium's id and the Isotropic `constant_medium` allotted).
#[derive(Clone, Copy, Debug, PartialEq)]
pub struct HitRecord {
    pub point: [f32; 3],
    pub normal: [f32; 3],
    pub t: f32,
    pub u: f32,
    pub v: f32,
    pub front_face: bool,
    pub material: MaterialId,
    pub hittable: HittableId,
}

/// A scene being recorded, then committed to the current CUDA device.  Not `Sync`: one caller per handle.
pub struct Scene {
    raw: *mut sys::shim_scene,
}
unsafe impl Send for Scene {}

impl Scene {
    pub fn new() -> Result<Scene> {
        let raw = unsafe { sys::shim_scene_create() };
        if raw.is_null() { Err(last_error(sys::SHIM_ERR_INVALID)) } else { Ok(Scene { raw }) }
    }
    pub fn as_raw(&self) -> *mut sys::shim_scene { self.raw }

    // textures/*.rs
    pub fn texture_solid(&mut self, r: f32, g: f32, b: f32) -> Result<TextureId> {
        check(unsafe { sys::shim_texture_solid(self.raw, r, g, b) }).map(TextureId)
    }
    pub fn texture_checker(&mut self, scale: f32, even: TextureId, odd: TextureId) -> Result<TextureId> {
        check(unsafe { sys::shim_texture_checker(self.raw, scale, even.0, odd.0) }).map(TextureId)
    }
    pub fn texture_marble(&mut self, scale: f32, perlin_seed: u32) -> Result<TextureId> {
        check(unsafe { sys::shim_texture_marble(self.raw, scale, perlin_seed) }).map(TextureId)
    }
    /// `rgb8`: tightly packed, `width * height * 3` bytes, top row first (image::RgbImage::as_raw()).
    pub fn texture_image(&mut self, rgb8: &[u8], width: u32, height: u32) -> Result<TextureId> {
        if rgb8.len() != width as usize * height as usize * 3 {
            return Err(Error { code: sys::SHIM_ERR_INVALID, message: "texture_image: buffer size".into() });
        }
        check(unsafe { sys::shim_texture_image(self.raw, rgb8.as_ptr(), width as c_int, height as c_int) }).map(TextureId)
    }

    // materials/*.rs
    pub fn lambertian(&mut self, albedo: TextureId) -> Result<MaterialId> {
        check(unsafe { sys::shim_material_lambertian(self.raw, albedo.0) }).map(MaterialId)
    }
    pub fn metal(&mut self, albedo: [f32; 3], fuzz: f32) -> Result<MaterialId> {
        check(unsafe { sys::shim_material_metal(self.raw, albedo[0], albedo[1], albedo[2], fuzz) }).map(MaterialId)
    }
    pub fn dielectric(&mut self, index_of_refraction: f32) -> Result<MaterialId> {
        check(unsafe { sys::shim_material_dielectric(self.raw, index_of_refraction) }).map(MaterialId)
    }
    pub fn diffuse_light(&mut self, emission: TextureId) -> Result<MaterialId> {
        check(unsafe { sys::shim_material_diffuse_light(self.raw, emission.0) }).map(MaterialId)
    }
    pub fn isotropic(&mut self, albedo: TextureId) -> Result<MaterialId> {
        check(unsafe { sys::shim_material_isotropic(self.raw, albedo.0) }).map(MaterialId)
    }

    // geometry/*.rs, hittable.rs, bvh.rs
    pub fn sphere(&mut self, center: [f32; 3], radius: f32, m: MaterialId) -> Result<HittableId> {
        check(unsafe { sys::shim_sphere(self.raw, center[0], center[1], center[2], radius, m.0) }).map(HittableId)
    }
    pub fn moving_sphere(&mut self, c0: [f32; 3], c1: [f32; 3], t0: f32, t1: f32, radius: f32, m: MaterialId) -> Result<HittableId> {
        check(unsafe { sys::shim_moving_sphere(self.raw, c0[0], c0[1], c0[2], c1[0], c1[1], c1[2], t0, t1, radius, m.0) }).map(HittableId)
    }
    pub fn xy_rect(&mut self, x0: f32, x1: f32, y0: f32, y1: f32, z: f32, m: MaterialId) -> Result<HittableId> {
        check(unsafe { sys::shim_xy_rect(self.raw, x0, x1, y0, y1, z, m.0) }).map(HittableId)
    }
    pub fn xz_rect(&mut self, x0: f32, x1: f32, z0: f32, z1: f32, y: f32, m: MaterialId) -> Result<HittableId> {
        check(unsafe { sys::shim_xz_rect(self.raw, x0, x1, z0, z1, y, m.0) }).map(HittableId)
    }
    pub fn yz_rect(&mut self, y0: f32, y1: f32, z0: f32, z1: f32, x: f32, m: MaterialId) -> Result<HittableId> {
        check(unsafe { sys::shim_yz_rect(self.raw, y0, y1, z0, z1, x, m.0) }).map(HittableId)
    }
    pub fn tri(&mut self, p0: [f32; 3], p1: [f32; 3], p2: [f32; 3], m: MaterialId) -> Result<HittableId> {
        let v = [p0[0], p0[1], p0[2], p1[0], p1[1], p1[2], p2[0], p2[1], p2[2]];
        check(unsafe { sys::shim_tri(self.raw, v.as_ptr(), m.0) }).map(HittableId)
    }
    pub fn cube(&mut self, min: [f32; 3], max: [f32; 3], m: MaterialId) -> Result<HittableId> {
        check(unsafe { sys::shim_cube(self.raw, min[0], min[1], min[2], max[0], max[1], max[2], m.0) }).map(HittableId)
    }
    pub fn list(&mut self) -> Result<HittableId> {
        check(unsafe { sys::shim_list_create(self.raw) }).map(HittableId)
    }
    pub fn list_add(&mut self, list: HittableId, h: HittableId) -> Result<()> {
        check(unsafe { sys::shim_list_add(self.raw, list.0, h.0) }).map(|_| ())
    }
    /// `xyz`: 9 floats per triangle (main.rs:745-789 `load_to_tris`); returns the id of the first triangle.
    pub fn tris_bulk(&mut self, xyz: &[f32], m: MaterialId, list: HittableId) -> Result<HittableId> {
        if xyz.len() % 9 != 0 {
            return Err(Error { code: sys::SHIM_ERR_INVALID, message: "tris_bulk: 9 floats per triangle".into() });
        }
        check(unsafe { sys::shim_tris_bulk(self.raw, xyz.as_ptr(), (xyz.len() / 9) as c_int, m.0, list.0) }).map(HittableId)
    }
    pub fn bvh(&mut self, list: HittableId, t0: f32, t1: f32, axis_seed: u64, with_predictor: bool) -> Result<HittableId> {
        check(unsafe { sys::shim_bvh(self.raw, list.0, t0, t1, axis_seed, with_predictor as c_int) }).map(HittableId)
    }
    /// A tree the caller built (`Bvh::nodes`): `left/right[i] >= 0` is a node index, `!id` a primitive child.
    pub fn bvh_from_nodes(&mut self, left: &[i32], right: &[i32], root: usize, t0: f32, t1: f32, with_predictor: bool) -> Result<HittableId> {
        if left.len() != right.len() {
            return Err(Error { code: sys::SHIM_ERR_INVALID, message: "bvh_from_nodes: left/right lengths differ".into() });
        }
        check(unsafe {
            sys::shim_bvh_from_nodes(self.raw, left.len() as c_int, left.as_ptr(), right.as_ptr(), root as c_int, t0, t1, with_predictor as c_int)
        })
        .map(HittableId)
    }
    pub fn translate(&mut self, h: HittableId, d: [f32; 3]) -> Result<HittableId> {
        check(unsafe { sys::shim_translate(self.raw, h.0, d[0], d[1], d[2]) }).map(HittableId)
    }
    pub fn rotate_y(&mut self, h: HittableId, degrees: f32) -> Result<HittableId> {
        check(unsafe { sys::shim_rotate_y(self.raw, h.0, degrees) }).map(HittableId)
    }
    pub fn constant_medium(&mut self, boundary: HittableId, density: f32, albedo: TextureId) -> Result<HittableId> {
        check(unsafe { sys::shim_constant_medium(self.raw, boundary.0, density, albedo.0) }).map(HittableId)
    }
    pub fn world_add(&mut self, h: HittableId) -> Result<()> {
        check(unsafe { sys::shim_world_add(self.raw, h.0) }).map(|_| ())
    }
    pub fn use_reference_bvh_on_device(&mut self, yes: bool) -> Result<()> {
        let v = if yes { sys::SHIM_DEVICE_BVH_REFERENCE } else { sys::SHIM_DEVICE_BVH_SAH };
        check(unsafe { sys::shim_scene_set_option(self.raw, sys::SHIM_OPT_DEVICE_BVH, v) }).map(|_| ())
    }
    pub fn commit(&mut self) -> Result<()> {
        check(unsafe { sys::shim_commit(self.raw) }).map(|_| ())
    }

    /// `Renderer::render` on the device: fills `out` (width * height * 3 linear RGB, row 0 = bottom row).
    pub fn render(&mut self, cam: &Camera, p: &RenderParams, out: &mut [f32]) -> Result<Stats> {
        if out.len() != p.width as usize * p.height as usize * 3 {
            return Err(Error { code: sys::SHIM_ERR_INVALID, message: "render: framebuffer size".into() });
        }
        let mut st = Stats::default();
        check(unsafe { sys::shim_render(self.raw, cam, p, out.as_mut_ptr(), &mut st) })?;
        Ok(st)
    }
    /// One image over several devices of this process (`shim_render_multi`): `devices` = CUDA ordinals (empty = all),
    /// `tiles` = shard by tile index instead of by sample range.  The combined mean lands in `out`.
    pub fn render_multi(&mut self, cam: &Camera, p: &RenderParams, devices: &[i32], tiles: bool, out: &mut [f32]) -> Result<Stats> {
        if out.len() != p.width as usize * p.height as usize * 3 {
            return Err(Error { code: sys::SHIM_ERR_INVALID, message: "render_multi: framebuffer size".into() });
        }
        let mut st = Stats::default();
        let mode = if tiles { sys::SHIM_SHARD_TILES } else { sys::SHIM_SHARD_SAMPLES };
        let ptr = if devices.is_empty() { std::ptr::null() } else { devices.as_ptr() };
        check(unsafe { sys::shim_render_multi(self.raw, cam, p, devices.len() as c_int, ptr, mode, out.as_mut_ptr(), &mut st) })?;
        Ok(st)
    }
    /// Gate-1 query: closest hit of `rays` (7 floats each: origin, direction, time) -> (primitive id or -1, t).
    pub fn trace_closest(&mut self, rays: &[f32], t_min: f32, t_max: f32, seed: u64) -> Result<(Vec<i32>, Vec<f32>)> {
        if rays.len() % 7 != 0 {
            return Err(Error { code: sys::SHIM_ERR_INVALID, message: "trace_closest: 7 floats per ray".into() });
        }
        let n = rays.len() / 7;
        let (mut prim, mut t) = (vec![-1i32; n], vec![f32::INFINITY; n]);
        check(unsafe {
            sys::shim_trace_closest(self.raw, rays.as_ptr(), n as i64, t_min, t_max, seed, prim.as_mut_ptr(), t.as_mut_ptr(), std::ptr::null_mut())
        })?;
        Ok((prim, t))
    }
    /// `Hittable::hit` on the world for each of `rays` (7 floats each) with the whole record; `None` = no hit, as
    /// `Option<HitRecord>` in the reference.  Same walk and Philox stream as `trace_closest`.
    pub fn trace_hit(&mut self, rays: &[f32], t_min: f32, t_max: f32, seed: u64) -> Result<Vec<Option<HitRecord>>> {
        if rays.len() % 7 != 0 {
            return Err(Error { code: sys::SHIM_ERR_INVALID, message: "trace_hit: 7 floats per ray".into() });
        }
        let n = rays.len() / 7;
        let mut raw = vec![sys::shim_hit_record::default(); n];
        check(unsafe {
            sys::shim_trace_hit(self.raw, rays.as_ptr(), n as i64, t_min, t_max, seed, raw.as_mut_ptr(), std::ptr::null_mut())
        })?;
        Ok(raw
            .iter()
            .map(|r| {
                (r.hittable >= 0).then(|| HitRecord {
                    point: r.point,
                    normal: r.normal,
                    t: r.t,
                    u: r.u,
                    v: r.v,
                    front_face: r.front_face != 0,
                    material: MaterialId(r.material),
                    hittable: HittableId(r.hittable),
                })
            })
            .collect())
    }
    /// Occlusion (any hit): is anything hit on each of `rays` (7 floats each) with t in [t_min, t_max]?  `true` exactly
    /// where `trace_closest` of the same rays and seed reports a hit; the walk stops at the first hit it finds.
    /// Visibility between points a and b: origin a, direction b - a, t in [1e-3, 1 - 1e-3].
    pub fn trace_occluded(&mut self, rays: &[f32], t_min: f32, t_max: f32, seed: u64) -> Result<Vec<bool>> {
        if rays.len() % 7 != 0 {
            return Err(Error { code: sys::SHIM_ERR_INVALID, message: "trace_occluded: 7 floats per ray".into() });
        }
        let n = rays.len() / 7;
        let mut occ = vec![0u8; n];
        check(unsafe {
            sys::shim_trace_occluded(self.raw, rays.as_ptr(), n as i64, t_min, t_max, seed, occ.as_mut_ptr(), std::ptr::null_mut())
        })?;
        Ok(occ.iter().map(|&o| o != 0).collect())
    }
}
impl Drop for Scene {
    fn drop(&mut self) {
        unsafe { sys::shim_scene_destroy(self.raw) }
    }
}

/// Page-locked framebuffer (`shim_host_alloc`): `Scene::render` copies device -> host straight into it.
pub struct HostFramebuffer {
    ptr: *mut f32,
    len: usize,
}
unsafe impl Send for HostFramebuffer {}
impl HostFramebuffer {
    pub fn new(width: usize, height: usize) -> Result<HostFramebuffer> {
        let len = width * height * 3;
        let ptr = unsafe { sys::shim_host_alloc(len) };
        if ptr.is_null() { Err(last_error(sys::SHIM_ERR_CUDA)) } else { Ok(HostFramebuffer { ptr, len }) }
    }
}
impl Deref for HostFramebuffer {
    type Target = [f32];
    fn deref(&self) -> &[f32] { unsafe { std::slice::from_raw_parts(self.ptr, self.len) } }
}
impl DerefMut for HostFramebuffer {
    fn deref_mut(&mut self) -> &mut [f32] { unsafe { std::slice::from_raw_parts_mut(self.ptr, self.len) } }
}
impl Drop for HostFramebuffer {
    fn drop(&mut self) {
        unsafe { sys::shim_host_free(self.ptr) }
    }
}

/// Releases every device's wavefront pool (`shim_shutdown`); scenes stay valid.  No render may be in flight.
pub fn shutdown() {
    unsafe { sys::shim_shutdown() };
}

/// `Renderer::write_ppm` (renderer.rs:107-127): P3 text, no gamma, top row first; `None` = stdout.
pub fn write_ppm(rgb: &[f32], width: usize, height: usize, path: Option<&str>) -> Result<i64> {
    if rgb.len() != width * height * 3 {
        return Err(Error { code: sys::SHIM_ERR_INVALID, message: "write_ppm: framebuffer size".into() });
    }
    let c = path.map(|p| CString::new(p).unwrap());
    let n = unsafe { sys::shim_write_ppm(rgb.as_ptr(), width as c_int, height as c_int, c.as_ref().map_or(std::ptr::null(), |s| s.as_ptr())) };
    if n < 0 { Err(last_error(n as c_int)) } else { Ok(n) }
}
