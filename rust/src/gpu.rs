//! src/gpu.rs — the crate-side binding of librtp_b200.so (include/rtp.h, ABI version 3). Add `pub mod gpu;` to src/lib.rs and
//! rust/build.rs as the crate's build.rs. NOT COMPILED in the image this was written in (no rustc): the struct layouts are
//! those of include/rtp.h, which tests/test_abi_host.py pins with a C program (sizeof / offsetof of every struct).
//!
//! It lives inside the crate because `Bvh`, `Material` and `Array2d` keep their fields private (bvh.rs:27-34,
//! material.rs:87-91, image.rs:11-15): the three `to_rtp` helpers at the bottom are the only code that reads them.
#![allow(non_camel_case_types)]
use crate::hittable::Hittable;
use crate::image::Tile;
use crate::material::{Emit, Material};
use crate::render::{Camera, Multisampler, SceneData};
use crate::texture::Texture;
use crate::utility::*;
use std::os::raw::{c_char, c_int};

#[repr(C)] #[derive(Clone, Copy)] pub struct rtp_ray { pub origin: [f64; 3], pub direction: [f64; 3], pub t_min: f64, pub t_max: f64 }
#[repr(C)] #[derive(Clone, Copy)] pub struct rtp_hit { pub leaf: u32, pub material: u32, pub t: f64 }
#[repr(C)] pub struct rtp_vertex { pub position: [f64; 3], pub normal: [f64; 3], pub uv: [f64; 2] } // == mesh::Vertex (needs #[repr(C)] there)
#[repr(C)] pub struct rtp_mesh { pub vertices: *const rtp_vertex, pub indices: *const u32, pub n_vertices: u32, pub n_indices: u32, pub material: u32, pub _pad: u32 }
/// kind: 0 sphere, 1 triangle, 2 nested List, 3 nested Bvh (mesh = first item in `nested`, triangle = item count)
#[repr(C)] #[derive(Clone, Copy)] pub struct rtp_hittable { pub kind: u32, pub material: u32, pub mesh: u32, pub triangle: u32, pub center: [f64; 3], pub radius: f64 }
#[repr(C)] #[derive(Clone, Copy)] pub struct rtp_emit { pub kind: u32, pub texture: u32, pub rgb: [f64; 3] }
#[repr(C)] pub struct rtp_material { pub scatter: u32, pub absorb: u32, pub absorb_texture: u32, pub _pad: u32, pub scatter_param: f64, pub absorb_rgb: [f64; 3], pub emit: rtp_emit }
#[repr(C)] pub struct rtp_texture { pub kind: u32, pub width: u32, pub height: u32, pub odd: u32, pub even: u32, pub _pad: u32, pub seed: i64, pub rgb: [f64; 3], pub rgba: *const u8 }
#[repr(C)] pub struct rtp_scene_desc { pub abi_version: u32, pub root_kind: u32, pub meshes: *const rtp_mesh, pub hittables: *const rtp_hittable,
    pub materials: *const rtp_material, pub textures: *const rtp_texture, pub n_meshes: u32, pub n_hittables: u32, pub n_materials: u32, pub n_textures: u32,
    pub background: rtp_emit, pub nested: *const rtp_hittable, pub n_nested: u32, pub _pad: u32 }
#[repr(C)] pub struct rtp_camera { pub aspect_ratio: f64, pub fov: f64, pub focal_dist: f64, pub lens_radius: f64, pub orientation: [f64; 9], pub position: [f64; 3] }
#[repr(C)] #[derive(Default)] pub struct rtp_render_params { pub width: u32, pub height: u32, pub num_samples: u32, pub max_bounce: u32, pub seed: u64,
    pub sample_begin: u32, pub sample_end: u32, pub tile_x: u32, pub tile_y: u32, pub tile_w: u32, pub tile_h: u32, pub flags: u32,
    pub device_mask: u32, pub row_offset: u32, pub row_stride: u32 }
#[repr(C)] #[derive(Default, Debug)] pub struct rtp_stats { pub rays: u64, pub paths: u64, pub node_visits: u64, pub triangle_tests: u64, pub sphere_tests: u64,
    pub leaf_gates: u64, pub conservative_violations: u64, pub device_ms: f64, pub kernel_launches: u64, pub order_rewalks: u64, pub trace_ms: f64, pub shade_ms: f64 }
#[repr(C)] #[derive(Default, Clone, Copy)] pub struct rtp_adaptive_params { pub min_samples: u32, pub max_samples: u32, pub batch: u32, pub _pad: u32,
    pub abs_tol: f64, pub rel_tol: f64 }
pub enum rtp_scene {}

#[link(name = "rtp_b200")]
extern "C" {
    fn rtp_init(device: c_int) -> c_int;
    fn rtp_device_count(count: *mut c_int) -> c_int;
    fn rtp_last_error() -> *const c_char;
    fn rtp_scene_create(desc: *const rtp_scene_desc, out: *mut *mut rtp_scene) -> c_int;
    fn rtp_scene_create_multi(desc: *const rtp_scene_desc, device_mask: u32, out: *mut *mut rtp_scene) -> c_int;
    fn rtp_scene_destroy(scene: *mut rtp_scene);
    fn rtp_trace_closest(scene: *mut rtp_scene, rays: *const rtp_ray, n: usize, hits: *mut rtp_hit, stats: *mut rtp_stats) -> c_int;
    fn rtp_trace_occluded(scene: *mut rtp_scene, rays: *const rtp_ray, n: usize, occluded: *mut u8, stats: *mut rtp_stats) -> c_int;
    fn rtp_render(scene: *mut rtp_scene, camera: *const rtp_camera, params: *const rtp_render_params,
                  rgb: *mut f64, foreground: *mut f64, stats: *mut rtp_stats) -> c_int;
    fn rtp_render_adaptive(scene: *mut rtp_scene, camera: *const rtp_camera, params: *const rtp_render_params, adaptive: *const rtp_adaptive_params,
                           rgb: *mut f64, foreground: *mut f64, samples: *mut u32, stats: *mut rtp_stats) -> c_int;
    fn rtp_render_aov(scene: *mut rtp_scene, camera: *const rtp_camera, params: *const rtp_render_params,
                      rgb: *mut f64, foreground: *mut f64, albedo: *mut f64, normal: *mut f64, stats: *mut rtp_stats) -> c_int;
}

type GpuResult<T> = Result<T, Box<dyn std::error::Error>>; // the crate's loaders return Result<_, Box<dyn Error>> (mesh.rs:145)

fn check(rc: c_int) -> GpuResult<()> {
    if rc == 0 { Ok(()) } else { Err(unsafe { std::ffi::CStr::from_ptr(rtp_last_error()) }.to_string_lossy().into_owned().into()) }
}

pub struct GpuScene(*mut rtp_scene);
unsafe impl Send for GpuScene {} // immutable after creation; rtp_* calls on one scene are serialised inside the library
unsafe impl Sync for GpuScene {}
impl Drop for GpuScene { fn drop(&mut self) { unsafe { rtp_scene_destroy(self.0) } } }

/// `Hittable` -> rtp_hittable; nested containers append their items to `nested` (inner containers first, so that a container's
/// run always lies before the container itself, which is what the library checks to rule out cycles)
fn flatten(h: &Hittable, nested: &mut Vec<rtp_hittable>) -> rtp_hittable {
    let zero = rtp_hittable { kind: 0, material: 0, mesh: 0, triangle: 0, center: [0.0; 3], radius: 0.0 };
    match h {
        Hittable::Sphere { center, radius, material } => rtp_hittable { kind: 0, material: material.0, center: [center.x, center.y, center.z], radius: *radius, ..zero },
        Hittable::Triangle { triangle, mesh } => rtp_hittable { kind: 1, mesh: mesh.0, triangle: triangle.0, ..zero },
        Hittable::List(items) => {
            let run: Vec<rtp_hittable> = items.iter().map(|x| flatten(x, nested)).collect();
            let first = nested.len() as u32;
            nested.extend(run.iter().copied());
            rtp_hittable { kind: 2, mesh: first, triangle: run.len() as u32, ..zero }
        }
        Hittable::Bvh(bvh) => { // needs `pub(crate) fn leaves(&self) -> &[Hittable]` next to the private field (bvh.rs:29)
            let run: Vec<rtp_hittable> = bvh.leaves().iter().map(|x| flatten(x, nested)).collect();
            let first = nested.len() as u32;
            nested.extend(run.iter().copied());
            rtp_hittable { kind: 3, mesh: first, triangle: run.len() as u32, ..zero }
        }
    }
}

impl GpuScene {
    /// `root` is the scene root handed to trace_path (example_scenes.rs:14-19): `Hittable::Bvh(Bvh::new(vec, ..))` or `Hittable::List(vec)`.
    /// device_mask = 0: one GPU (device 0); otherwise bit d = CUDA device d holds a replica and render / hit_batch fan out.
    pub fn new(root: &Hittable, data: &SceneData, background: &Emit, device_mask: u32) -> GpuResult<Self> {
        let (items, as_bvh): (&[Hittable], bool) = match root {
            Hittable::Bvh(bvh) => (bvh.leaves(), true),
            Hittable::List(v) => (v.as_slice(), false),
            other => (std::slice::from_ref(other), false),
        };
        let mut nested = Vec::new();
        let hs: Vec<rtp_hittable> = items.iter().map(|h| flatten(h, &mut nested)).collect();
        let meshes: Vec<rtp_mesh> = data.mesh_table.iter().map(|m| rtp_mesh {
            vertices: m.vertices.as_ptr() as *const rtp_vertex, indices: m.indices.as_ptr(),
            n_vertices: m.vertices.len() as u32, n_indices: m.indices.len() as u32, material: m.material.0, _pad: 0 }).collect();
        let materials: Vec<rtp_material> = data.material_table.iter().map(Material::to_rtp).collect();
        let textures: Vec<rtp_texture> = data.texture_table.iter().map(Texture::to_rtp).collect();
        let desc = rtp_scene_desc { abi_version: 3, root_kind: if as_bvh { 0 } else { 1 }, meshes: meshes.as_ptr(), hittables: hs.as_ptr(),
            materials: materials.as_ptr(), textures: textures.as_ptr(), n_meshes: meshes.len() as u32, n_hittables: hs.len() as u32,
            n_materials: materials.len() as u32, n_textures: textures.len() as u32, background: background.to_rtp(),
            nested: nested.as_ptr(), n_nested: nested.len() as u32, _pad: 0 };
        let mut scene = std::ptr::null_mut();
        if device_mask == 0 {
            check(unsafe { rtp_init(0) })?;
            check(unsafe { rtp_scene_create(&desc, &mut scene) })?; // inputs are copied; the Vecs above may drop now
        } else {
            check(unsafe { rtp_scene_create_multi(&desc, device_mask, &mut scene) })?;
        }
        Ok(GpuScene(scene))
    }

    pub fn device_count() -> GpuResult<u32> { let mut n = 0; check(unsafe { rtp_device_count(&mut n) })?; Ok(n as u32) }

    /// Batched `Hittable::hit` on the root (bvh.rs:121-124 / hittable.rs:110-120): `hits[k].leaf` = index of the root item that holds
    /// the winner (u32::MAX on a miss), `.material` its MaterialId, `.t` = Hit::t.
    pub fn hit_batch(&self, rays: &[Ray]) -> GpuResult<Vec<rtp_hit>> {
        let rs = Self::rays(rays);
        let mut hits = vec![rtp_hit { leaf: u32::MAX, material: u32::MAX, t: f64::INFINITY }; rs.len()];
        check(unsafe { rtp_trace_closest(self.0, rs.as_ptr(), rs.len(), hits.as_mut_ptr(), std::ptr::null_mut()) })?;
        Ok(hits)
    }

    /// `scene.hit(ray).is_some()` (hittable.rs:18-25, bvh.rs:121-124) for a batch: true iff the ray hits anything with
    /// t_min <= t <= t_max, bit for bit `hit_batch(..)[k].leaf != u32::MAX`; the walk stops at the first accepted leaf.
    pub fn occluded(&self, rays: &[Ray]) -> GpuResult<Vec<bool>> {
        let rs = Self::rays(rays);
        let mut occ = vec![0u8; rs.len()];
        check(unsafe { rtp_trace_occluded(self.0, rs.as_ptr(), rs.len(), occ.as_mut_ptr(), std::ptr::null_mut()) })?;
        Ok(occ.into_iter().map(|b| b != 0).collect())
    }

    fn rays(rays: &[Ray]) -> Vec<rtp_ray> {
        rays.iter().map(|r| rtp_ray { origin: [r.origin.x, r.origin.y, r.origin.z],
            direction: [r.direction.x, r.direction.y, r.direction.z], t_min: r.t_min, t_max: r.t_max }).collect()
    }

    fn camera(camera: &Camera) -> rtp_camera {
        let t = &camera.transformation;
        let m = t.orientation; // Rmat3, columns x, y, z (utility.rs:176)
        rtp_camera { aspect_ratio: camera.aspect_ratio, fov: camera.fov, focal_dist: camera.focal_dist, lens_radius: camera.lens_radius,
            orientation: [m[(0, 0)], m[(1, 0)], m[(2, 0)], m[(0, 1)], m[(1, 1)], m[(2, 1)], m[(0, 2)], m[(1, 2)], m[(2, 2)]],
            position: [t.position.x, t.position.y, t.position.z] }
    }

    /// main.rs:61-92 for one tile; writes `Σ/num_samples` into the caller's full-frame buffers (row j = 0 at the bottom).
    pub fn render_tile(&self, camera: &Camera, sampler: &Multisampler, tile: &Tile, max_bounce: u32, seed: u64,
                       rgb: &mut [f64], foreground: &mut [f64]) -> GpuResult<rtp_stats> {
        let p = rtp_render_params { width: sampler.width, height: sampler.height, num_samples: sampler.num_samples, max_bounce, seed,
            sample_begin: 0, sample_end: sampler.num_samples, tile_x: tile.offset_i, tile_y: tile.offset_j, tile_w: tile.width, tile_h: tile.height,
            ..Default::default() };
        let mut stats = rtp_stats::default();
        check(unsafe { rtp_render(self.0, &Self::camera(camera), &p, rgb.as_mut_ptr(), foreground.as_mut_ptr(), &mut stats) })?;
        Ok(stats)
    }

    /// The whole worker phase of main.rs:46-98 in one call: every device of the scene renders its share of the rows.
    pub fn render_frame(&self, camera: &Camera, sampler: &Multisampler, max_bounce: u32, seed: u64) -> GpuResult<(Vec<f64>, Vec<f64>, rtp_stats)> {
        let npx = (sampler.width * sampler.height) as usize;
        let (mut rgb, mut fg) = (vec![0.0; 3 * npx], vec![0.0; npx]);
        let p = rtp_render_params { width: sampler.width, height: sampler.height, num_samples: sampler.num_samples, max_bounce, seed,
            sample_begin: 0, sample_end: sampler.num_samples, ..Default::default() };
        let mut stats = rtp_stats::default();
        check(unsafe { rtp_render(self.0, &Self::camera(camera), &p, rgb.as_mut_ptr(), fg.as_mut_ptr(), &mut stats) })?;
        Ok((rgb, fg, stats))
    }

    /// render_frame plus the guide buffers of a denoiser: per pixel the mean over its samples of the first vertex's
    /// `Absorb::evaluate` (material.rs:74-81) and `Hit::normal` (not flipped, not renormalised; (0, 0, 0) for a miss).
    /// Returns (rgb, foreground, albedo, normal, stats); rgb and foreground are render_frame's bits.
    pub fn render_frame_aov(&self, camera: &Camera, sampler: &Multisampler, max_bounce: u32, seed: u64)
                            -> GpuResult<(Vec<f64>, Vec<f64>, Vec<f64>, Vec<f64>, rtp_stats)> {
        let npx = (sampler.width * sampler.height) as usize;
        let (mut rgb, mut fg, mut albedo, mut normal) = (vec![0.0; 3 * npx], vec![0.0; npx], vec![0.0; 3 * npx], vec![0.0; 3 * npx]);
        let p = rtp_render_params { width: sampler.width, height: sampler.height, num_samples: sampler.num_samples, max_bounce, seed,
            sample_begin: 0, sample_end: sampler.num_samples, ..Default::default() };
        let mut stats = rtp_stats::default();
        check(unsafe { rtp_render_aov(self.0, &Self::camera(camera), &p, rgb.as_mut_ptr(), fg.as_mut_ptr(), albedo.as_mut_ptr(),
                                      normal.as_mut_ptr(), &mut stats) })?;
        Ok((rgb, fg, albedo, normal, stats))
    }
}

// ---- the three accessors the private fields require (each next to its type in the real patch) ---------------------------------
impl Material { // material.rs:87-100
    pub(crate) fn to_rtp(&self) -> rtp_material {
        use crate::material::{Absorb, Scatter};
        let (scatter, scatter_param) = match self.scatter { Scatter::None => (0, 0.0), Scatter::Lambert => (1, 0.0),
            Scatter::Metal { fuzziness } => (2, fuzziness), Scatter::Dielectric { refraction_index } => (3, refraction_index) };
        let (absorb, absorb_rgb, absorb_texture) = match &self.absorb { Absorb::BlackBody => (0, [0.0; 3], 0), Absorb::WhiteBody => (1, [0.0; 3], 0),
            Absorb::Albedo(c) => (2, [c.x, c.y, c.z], 0), Absorb::AlbedoMap(t) => (3, [0.0; 3], t.0) };
        rtp_material { scatter, absorb, absorb_texture, _pad: 0, scatter_param, absorb_rgb, emit: self.emit.to_rtp() }
    }
}
impl Emit { // material.rs:40-46
    pub(crate) fn to_rtp(&self) -> rtp_emit {
        match self { Emit::None => rtp_emit { kind: 0, texture: 0, rgb: [0.0; 3] }, Emit::DebugNormals => rtp_emit { kind: 1, texture: 0, rgb: [0.0; 3] },
            Emit::Color(c) => rtp_emit { kind: 2, texture: 0, rgb: [c.x, c.y, c.z] }, Emit::SkyGradient => rtp_emit { kind: 3, texture: 0, rgb: [0.0; 3] },
            Emit::SkySphere(t) => rtp_emit { kind: 4, texture: t.0, rgb: [0.0; 3] } }
    }
}
impl Texture { // texture.rs:10-18; Image borrows the texel storage of Array2d<[u8; 4]> (row 0 = bottom, image.rs:31-33)
    pub(crate) fn to_rtp(&self) -> rtp_texture {
        let z = rtp_texture { kind: 0, width: 0, height: 0, odd: 0, even: 0, _pad: 0, seed: 0, rgb: [0.0; 3], rgba: std::ptr::null() };
        match self { Texture::Missing => z, Texture::DebugUVs => rtp_texture { kind: 1, ..z }, Texture::Solid(c) => rtp_texture { kind: 2, rgb: [c.x, c.y, c.z], ..z },
            Texture::Image(img) => rtp_texture { kind: 3, width: img.width() as u32, height: img.height() as u32, rgba: img.as_ptr() as *const u8, ..z },
            Texture::Checker { odd, even } => rtp_texture { kind: 4, odd: odd.0, even: even.0, ..z },
            Texture::Noise { seed } => rtp_texture { kind: 5, seed: *seed as i64, ..z }, Texture::Perlin { seed } => rtp_texture { kind: 6, seed: *seed as i64, ..z } }
    }
}
