//! src/pathtracer/gpu/b200.rs — the B200 path behind pathtracer-rs's own interfaces (feature "b200").
//!
//! Drop-in points (reference file:line):
//!   * `PathIntegrator::render(&self, &Camera, &RenderScene)`      src/pathtracer/integrator.rs:536
//!   * `RenderScene::{intersect, intersect_p}`                     src/pathtracer/mod.rs:92-98
//!   * the unused `OptixAccelerator::new(&RenderScene)` hook       src/pathtracer/gpu/optix.rs:160
//! The intrusive part is small and additive: read-only exporters on the reference's own types
//! (`reference_additions.rs`: `BVH::export_flat`, `Texture::export`, `Material::export`, `Light::export`, a few
//! accessors), because accelerator.rs, primitive.rs, shape.rs, texture.rs, material/*.rs and light.rs keep the fields
//! private.  `tables.rs` interns meshes / materials / textures / lights into the flat pools; `ffi.rs` is generated from
//! include/ptrs_b200.h.  Written against the reference's types and NOT compiled: the pathtracer-b200 image has no Rust
//! toolchain; `examples/c_abi_shim.c` fills a PtrsSceneDesc the same way from plain C and runs in the GPU tests.
use super::ffi;
use super::tables::Tables;
use crate::common::{film::Film, Camera};
use crate::pathtracer::{accelerator::LinearBVHNode, RenderScene};
use std::ffi::CStr;

#[derive(Debug)]
pub struct B200Error {
    pub code: i32,
    pub message: String,
}

fn check(code: i32) -> Result<(), B200Error> {
    if code == ffi::PTRS_OK {
        return Ok(());
    }
    let message = unsafe { CStr::from_ptr(ffi::ptrs_last_error()) }.to_string_lossy().into_owned();
    Err(B200Error { code, message })
}

/// Flat copy of a `RenderScene` in the layout of `PtrsSceneDesc`; owns the arrays the descriptor points into.
#[derive(Default)]
pub struct FlatScene {
    pub nodes: Vec<ffi::PtrsBvhNode>,
    pub prim_vertex: Vec<u32>,
    pub prim_mesh: Vec<i32>,
    pub prim_material: Vec<i32>,
    pub prim_area_light: Vec<i32>,
    pub pos: Vec<f32>,
    pub normal: Vec<f32>,
    pub tangent: Vec<f32>,
    pub uv: Vec<f32>,
    pub meshes: Vec<ffi::PtrsMesh>,
    pub materials: Vec<ffi::PtrsMaterial>,
    pub textures: Vec<ffi::PtrsTexture>,
    pub mipmaps: Vec<ffi::PtrsMipMap>,
    pub texels: Vec<f32>,
    pub lights: Vec<ffi::PtrsLight>,
    pub infinite_lights: Vec<i32>,
    pub envs: Vec<ffi::PtrsEnvLight>,
    env_arrays: Vec<Vec<f32>>, // Distribution2D func / cdf / func_int vectors behind `envs`
}

impl FlatScene {
    /// `BVH::export_flat()` yields the node array verbatim — `LinearBVHNode` is `#[repr(C, align(32))]` and has
    /// the layout of `PtrsBvhNode` (accelerator.rs:83-95) — and the primitives in `BVH::primitives` order.
    pub fn from_render_scene(scene: &RenderScene) -> Self {
        let mut flat = FlatScene::default();
        let (nodes, prims) = scene.bvh().export_flat(); // reference_additions.rs
        flat.nodes = nodes.iter().map(node_to_ffi).collect();
        let mut tables = Tables::new(&scene.meshes, &scene.lights, &scene.infinite_lights);
        for (i, prim) in prims.iter().enumerate() {
            let tri = prim.get_shape();
            let base = tables.vertex_base(tri.mesh());
            flat.prim_vertex.extend(tri.indices().iter().map(|v| base + *v));
            flat.prim_mesh.push(tables.mesh_id(tri.mesh()));
            flat.prim_material.push(tables.material_id(prim.get_material_arc()));
            flat.prim_area_light.push(prim.get_area_light().map_or(-1, |l| tables.light_id(l)));
            if prim.get_area_light().is_some() {
                tables.note_prim(tri, i);
            }
        }
        tables.write_pools(&mut flat); // pos / normal / s / uv, materials, textures + MIP pyramids, lights, envs
        flat
    }

    /// InfiniteAreaLight (light.rs:321-399): the transforms, the map's pyramid and the Distribution2D exactly as the
    /// reference built them (sampling.rs:185-209).  Leaving the five arrays empty instead makes the library build the
    /// distribution on the device (include/ptrs_b200.h, PtrsEnvLight).
    pub fn push_env(
        &mut self,
        tables: &mut Tables,
        light_to_world: &na::Projective3<f32>,
        world_to_light: &na::Projective3<f32>,
        l_map: &crate::pathtracer::texture::MIPMap<crate::common::spectrum::Spectrum>,
        distribution: &crate::pathtracer::sampling::Distribution2D,
    ) -> i32 {
        let row_major = |m: &na::Projective3<f32>| {
            let mut o = [0f32; 16];
            for r in 0..4 {
                for c in 0..4 {
                    o[4 * r + c] = m.matrix()[(r, c)];
                }
            }
            o
        };
        let (rows, marginal) = distribution.parts();
        let (marg_func, marg_cdf, marg_func_int) = marginal.parts();
        let nv = rows.len();
        let nu = rows[0].parts().0.len();
        let mut cond_func = Vec::with_capacity(nu * nv);
        let mut cond_cdf = Vec::with_capacity((nu + 1) * nv);
        let mut cond_func_int = Vec::with_capacity(nv);
        for row in rows {
            let (f, c, fi) = row.parts();
            cond_func.extend_from_slice(f);
            cond_cdf.extend_from_slice(c);
            cond_func_int.push(fi);
        }
        let base = self.env_arrays.len();
        self.env_arrays.extend([cond_func, cond_cdf, cond_func_int, marg_func.to_vec(), marg_cdf.to_vec()]);
        let a = &self.env_arrays[base..];
        self.envs.push(ffi::PtrsEnvLight {
            light_to_world: row_major(light_to_world),
            world_to_light: row_major(world_to_light),
            mip: tables.push_env_mip(l_map),
            nu: nu as i32,
            nv: nv as i32,
            pad: 0,
            cond_func: a[0].as_ptr(),
            cond_cdf: a[1].as_ptr(),
            cond_func_int: a[2].as_ptr(),
            marg_func: a[3].as_ptr(),
            marg_cdf: a[4].as_ptr(),
            marg_func_int,
            pad2: 0.0,
        });
        self.envs.len() as i32 - 1
    }

    pub fn desc(&self) -> ffi::PtrsSceneDesc {
        fn ptr<T>(v: &[T]) -> *const T {
            if v.is_empty() { std::ptr::null() } else { v.as_ptr() }
        }
        ffi::PtrsSceneDesc {
            abi_version: ffi::PTRS_ABI_VERSION,
            n_nodes: self.nodes.len() as u32,
            nodes: ptr(&self.nodes),
            n_prims: self.prim_mesh.len() as u32,
            prim_vertex: ptr(&self.prim_vertex),
            prim_mesh: ptr(&self.prim_mesh),
            prim_material: ptr(&self.prim_material),
            prim_area_light: ptr(&self.prim_area_light),
            n_verts: (self.pos.len() / 3) as u32,
            pos: ptr(&self.pos),
            normal: ptr(&self.normal),
            tangent: ptr(&self.tangent),
            uv: ptr(&self.uv),
            n_meshes: self.meshes.len() as u32,
            meshes: ptr(&self.meshes),
            n_materials: self.materials.len() as u32,
            materials: ptr(&self.materials),
            n_textures: self.textures.len() as u32,
            textures: ptr(&self.textures),
            n_mipmaps: self.mipmaps.len() as u32,
            mipmaps: ptr(&self.mipmaps),
            n_texels: self.texels.len() as u64,
            texels: ptr(&self.texels),
            n_lights: self.lights.len() as u32,
            lights: ptr(&self.lights),
            n_infinite_lights: self.infinite_lights.len() as u32,
            infinite_lights: ptr(&self.infinite_lights),
            n_envs: self.envs.len() as u32,
            envs: ptr(&self.envs),
        }
    }
}

fn node_to_ffi(n: &LinearBVHNode) -> ffi::PtrsBvhNode {
    // same 32 bytes; spelled out so that a layout change on either side fails to compile instead of corrupting
    ffi::PtrsBvhNode {
        bounds_min: [n.bounds.p_min.x, n.bounds.p_min.y, n.bounds.p_min.z],
        bounds_max: [n.bounds.p_max.x, n.bounds.p_max.y, n.bounds.p_max.z],
        offset: n.offset(),
        n_prims: n.num_prims,
        axis: n.axis,
        pad: 0,
    }
}

/// Device copy of a scene: what `RenderScene` holds (`Box<BVH>`, lights) on the GPU.
pub struct B200Scene {
    handle: *mut ffi::PtrsScene,
}
unsafe impl Send for B200Scene {}

impl B200Scene {
    /// Reference-built BVH (bit-identical hit order to the CPU path).
    pub fn new(scene: &RenderScene) -> Result<Self, B200Error> {
        let flat = FlatScene::from_render_scene(scene);
        let mut handle = std::ptr::null_mut();
        check(unsafe { ffi::ptrs_scene_create(&flat.desc(), &mut handle) })?;
        Ok(Self { handle }) // the library copied everything: `flat` may drop here
    }
    /// Skips `BVH::new` on the host: the tree is built on the device in milliseconds.
    pub fn new_device_bvh(flat: &FlatScene) -> Result<Self, B200Error> {
        let mut handle = std::ptr::null_mut();
        check(unsafe { ffi::ptrs_scene_create_device_bvh(&flat.desc(), &mut handle) })?;
        Ok(Self { handle })
    }
    /// `RenderScene::intersect` over a batch (mod.rs:92-94): prim == -1 is a miss.
    pub fn intersect(&self, rays: &[ffi::PtrsRay]) -> Result<Vec<ffi::PtrsHit>, B200Error> {
        let mut hits = vec![ffi::PtrsHit { prim: -1, t: 0.0, b0: 0.0, b1: 0.0, b2: 0.0 }; rays.len()];
        check(unsafe { ffi::ptrs_intersect(self.handle, rays.as_ptr(), rays.len(), hits.as_mut_ptr()) })?;
        Ok(hits)
    }
    /// `RenderScene::intersect_p` over a batch (mod.rs:96-98).
    pub fn intersect_p(&self, rays: &[ffi::PtrsRay]) -> Result<Vec<bool>, B200Error> {
        let mut occ = vec![0u8; rays.len()];
        check(unsafe { ffi::ptrs_intersect_p(self.handle, rays.as_ptr(), rays.len(), occ.as_mut_ptr()) })?;
        Ok(occ.into_iter().map(|o| o != 0).collect())
    }
}

impl Drop for B200Scene {
    fn drop(&mut self) {
        unsafe { ffi::ptrs_scene_destroy(self.handle) };
    }
}

pub fn camera_to_ffi(camera: &Camera) -> ffi::PtrsCamera {
    let q = camera.cam_to_world.rotation.coords; // (i, j, k, w)
    let t = camera.cam_to_world.translation.vector;
    let r2s = camera.raster_to_screen.matrix();
    let mut raster_to_screen = [0f32; 16];
    for r in 0..4 {
        for c in 0..4 {
            raster_to_screen[4 * r + c] = r2s[(r, c)]; // row-major
        }
    }
    let p = camera.cam_to_screen.as_matrix();
    ffi::PtrsCamera {
        rot: [q.x, q.y, q.z, q.w],
        trans: [t.x, t.y, t.z],
        pad0: 0.0,
        raster_to_screen,
        persp: [p[(0, 0)], p[(1, 1)], p[(2, 2)], p[(2, 3)]],
        dx_camera: [camera.dx_camera.x, camera.dx_camera.y, camera.dx_camera.z],
        dy_camera: [camera.dy_camera.x, camera.dy_camera.y, camera.dy_camera.z],
        width: camera.film.resolution.x as i32,
        height: camera.film.resolution.y as i32,
    }
}

/// What `PathIntegrator::render` does with the feature on (integrator.rs:536): same arguments, accumulates into
/// `camera.film`, logs instead of failing.
pub fn render(
    log: &slog::Logger,
    gpu: &B200Scene,
    camera: &Camera,
    spp: usize,
    max_depth: i32,
    rr_threshold: f32,
    rr_start_depth: i32,
    rr_enable: bool,
) {
    render_region(log, gpu, camera, None, spp, max_depth, rr_threshold, rr_start_depth, rr_enable)
}

/// The same restricted to a rectangle of sample positions `[x0, y0, x1, y1]` (half-open, inside the film's sample
/// bounds; `None` = all of them), e.g. one tile of integrator.rs:545-637 or, with `ptrs_film_region_sample_rect`, the
/// samples that complete a pixel crop.  Only film pixels within the rectangle's filter footprint change.
pub fn render_region(
    log: &slog::Logger,
    gpu: &B200Scene,
    camera: &Camera,
    sample_rect: Option<[i32; 4]>,
    spp: usize,
    max_depth: i32,
    rr_threshold: f32,
    rr_start_depth: i32,
    rr_enable: bool,
) {
    let mut params: ffi::PtrsRenderParams = unsafe { std::mem::zeroed() };
    unsafe { ffi::ptrs_render_params_default(&mut params) };
    params.spp = spp as i32; // rounded up to a power of two inside, like sobol.rs:37
    params.max_depth = max_depth;
    params.rr_threshold = rr_threshold;
    params.rr_start_depth = rr_start_depth;
    params.rr_enable = rr_enable as i32;
    let cam = camera_to_ffi(camera);
    let (w, h) = (cam.width, cam.height);
    let mut film = std::ptr::null_mut();
    let result = check(unsafe { ffi::ptrs_film_create(w, h, &mut film) })
        .and_then(|_| {
            check(unsafe {
                match sample_rect {
                    Some(r) => ffi::ptrs_render_region(gpu.handle, &cam, &params, r.as_ptr(), film, std::ptr::null_mut()),
                    None => ffi::ptrs_render(gpu.handle, &cam, &params, film, std::ptr::null_mut()),
                }
            })
        })
        .and_then(|_| {
            let mut rgbw = vec![0f32; (w * h * 4) as usize];
            check(unsafe { ffi::ptrs_film_download(film, rgbw.as_mut_ptr()) }).map(|_| rgbw)
        });
    match result {
        Ok(rgbw) => merge_into_film(&camera.film, &rgbw),
        Err(e) => error!(log, "B200 render failed ({}): {}", e.code, e.message),
    }
    if !film.is_null() {
        unsafe { ffi::ptrs_film_destroy(film) };
    }
}

/// `Film::merge_film_tile` for the whole image (film.rs:213-228): the device film holds the same two sums.
fn merge_into_film(film: &Film, rgbw: &[f32]) {
    let mut pixels = film.pixels.write().unwrap();
    for (pixel, src) in pixels.iter_mut().zip(rgbw.chunks_exact(4)) {
        pixel.xyz[0] += src[0];
        pixel.xyz[1] += src[1];
        pixel.xyz[2] += src[2];
        pixel.filter_weight_sum += src[3];
    }
}
