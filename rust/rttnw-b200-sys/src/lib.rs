//! Host side of the B200 backend for rttnw: raw bindings (`ffi`) and, on top of them, a scene builder
//! the reference's trait objects write themselves into (`SceneBuilder`) and a renderer (`Gpu`).
//!
//! The reference's hot path is the closure of `render()` (src/main.rs:199-229): for every pixel and
//! sample, `camera.ray` + `color(ray, background, &world, 50)`. With this crate that closure becomes
//! `Gpu::render(&desc, width, height, samples) -> Vec<u8>`; everything around it (scene table, image
//! save, CLI) stays as it is. INTEGRATION.md shows the three edits inside the reference's tree:
//! one `describe` method per trait, `BvhTree` remembering its list, and the new `render()` body.
//!
//! Modules: `ffi` (raw bindings), `math` (the reference's scene API as description-only types: every `Hittable`,
//! `Material` and `Texture` of src/math/*.rs with a `describe` method), `scenes` (the reference's own scenes.rs,
//! included and compiled against `math`), `render` (the scene table and `render()`).
//!
//! NOT BUILT in this repository's image (no Rust toolchain): reviewed source only.
pub mod ffi;
pub mod math;
pub mod render;
pub mod scenes;

pub use render::{render, render_world, scene_setup, shard_spp};

use std::collections::HashMap;
use std::ffi::CStr;
use std::os::raw::c_void;
use std::ptr;

/// An error reported by the library (`rtx_last_error`).
#[derive(Debug)]
pub struct RtxError {
    pub status: i32,
    pub message: String,
}

pub(crate) fn check(status: i32) -> Result<(), RtxError> {
    if status == ffi::RTX_OK {
        return Ok(());
    }
    let message = unsafe {
        let p = ffi::rtx_last_error();
        if p.is_null() { String::new() } else { CStr::from_ptr(p).to_string_lossy().into_owned() }
    };
    Err(RtxError { status, message })
}

/// Collects the plain-data description `rtx_scene_create` consumes. Shared objects (`Arc`) are
/// emitted once: `material_of` / `texture_of` / `node_of` key them by pointer identity.
#[derive(Default)]
pub struct SceneBuilder {
    nodes: Vec<ffi::rtx_node>,
    children: Vec<i32>,
    materials: Vec<ffi::rtx_material>,
    textures: Vec<ffi::rtx_texture>,
    perlins: Vec<ffi::rtx_perlin>,
    images: Vec<(i32, i32, Option<Vec<u8>>)>,
    seen: HashMap<(u8, usize), i32>,
    unsupported: Option<&'static str>,
}

impl SceneBuilder {
    pub fn new() -> Self {
        Self::default()
    }

    /// Index of an already described shared object (kind: 0 node, 1 material, 2 texture), by address.
    pub fn seen<T: ?Sized>(&self, kind: u8, object: *const T) -> Option<i32> {
        self.seen.get(&(kind, object as *const u8 as usize)).copied()
    }
    pub fn remember<T: ?Sized>(&mut self, kind: u8, object: *const T, index: i32) -> i32 {
        self.seen.insert((kind, object as *const u8 as usize), index);
        index
    }

    /// A leaf or wrapper node; `f` follows the per-kind layout documented in rttnw_b200.h.
    pub fn node(&mut self, kind: i32, material: i32, child: i32, f: [f64; 10]) -> i32 {
        self.nodes.push(ffi::rtx_node { kind, material, child, n_children: 0, f });
        self.nodes.len() as i32 - 1
    }
    /// A `List` (kind RTX_NODE_LIST) or `BvhTree` (RTX_NODE_BVH) over already described items.
    pub fn list(&mut self, kind: i32, items: &[i32]) -> i32 {
        let first = self.children.len() as i32;
        self.children.extend_from_slice(items);
        self.nodes.push(ffi::rtx_node { kind, material: -1, child: first, n_children: items.len() as i32, f: [0.0; 10] });
        self.nodes.len() as i32 - 1
    }
    pub fn material(&mut self, kind: i32, texture: i32, albedo: [f64; 3], param: f64) -> i32 {
        self.materials.push(ffi::rtx_material { kind, texture, albedo, param });
        self.materials.len() as i32 - 1
    }
    pub fn solid(&mut self, rgb: [f64; 3]) -> i32 {
        self.texture(ffi::RTX_TEX_SOLID, 0, 0, [rgb[0], rgb[1], rgb[2], 0.0])
    }
    pub fn texture(&mut self, kind: i32, a: i32, b: i32, f: [f64; 4]) -> i32 {
        self.textures.push(ffi::rtx_texture { kind, a, b, _pad: 0, f });
        self.textures.len() as i32 - 1
    }
    /// `Perlin` (noise.rs:5-29): 256 gradient vectors and the three permutations, as generated.
    pub fn perlin(&mut self, ranvec: &[[f64; 3]], perm_x: &[usize], perm_y: &[usize], perm_z: &[usize]) -> i32 {
        let mut p = ffi::rtx_perlin { ranvec: [[0.0; 3]; 256], perm_x: [0; 256], perm_y: [0; 256], perm_z: [0; 256] };
        for i in 0..256 {
            p.ranvec[i] = ranvec[i];
            p.perm_x[i] = perm_x[i] as i32;
            p.perm_y[i] = perm_y[i] as i32;
            p.perm_z[i] = perm_z[i] as i32;
        }
        self.perlins.push(p);
        self.perlins.len() as i32 - 1
    }
    /// `ImageTexture` (texture.rs:61-75): the decoded RGBA8 pixels, or None when the load failed (cyan).
    pub fn image(&mut self, width: u32, height: u32, rgba: Option<Vec<u8>>) -> i32 {
        self.images.push((width as i32, height as i32, rgba));
        self.images.len() as i32 - 1
    }
    /// The default of `Hittable::describe` etc.: a user type with no device counterpart. The render
    /// then fails loudly instead of silently dropping the object.
    pub fn unsupported(&mut self, type_name: &'static str) -> i32 {
        self.unsupported.get_or_insert(type_name);
        -1
    }
}

/// One CUDA device: context, and the renders made through it.
pub struct Gpu {
    ctx: *mut ffi::rtx_ctx,
}

impl Gpu {
    pub fn new(device: i32) -> Result<Gpu, RtxError> {
        let mut ctx = ptr::null_mut();
        check(unsafe { ffi::rtx_ctx_create(device, ptr::null_mut(), &mut ctx) })?;
        Ok(Gpu { ctx })
    }

    /// The replacement of the pixel loop of `render()` (src/main.rs:199-229): `samples` paths per pixel
    /// of the scene in `b` (root node `root`), sqrt gamma, RGBA8, top row first — what the reference
    /// hands to `image::save_buffer`.
    #[allow(clippy::too_many_arguments)]
    pub fn render(&self, b: &SceneBuilder, root: i32, camera: ffi::rtx_camera, background: [f64; 3], width: u32, height: u32,
                  samples: usize, seed: u64) -> Result<Vec<u8>, RtxError> {
        if let Some(name) = b.unsupported {
            return Err(RtxError { status: -5, message: format!("{} has no device counterpart", name) });
        }
        let images: Vec<ffi::rtx_image> = b.images.iter()
            .map(|(w, h, px)| ffi::rtx_image { width: *w, height: *h, rgba: px.as_ref().map_or(ptr::null(), |v| v.as_ptr()) })
            .collect();
        let desc = ffi::rtx_scene_desc {
            nodes: b.nodes.as_ptr(), n_nodes: b.nodes.len() as i32, root,
            children: b.children.as_ptr(), n_children: b.children.len() as i32, n_materials: b.materials.len() as i32,
            materials: b.materials.as_ptr(), textures: b.textures.as_ptr(),
            n_textures: b.textures.len() as i32, n_perlins: b.perlins.len() as i32, perlins: b.perlins.as_ptr(),
            images: images.as_ptr(), n_images: images.len() as i32, _pad: 0,
            background, camera,
        };
        self.render_desc(&desc, width, height, samples, seed)
    }

    /// The same for a ready-made description (e.g. `rtx_builtin_scene`).
    pub fn render_desc(&self, desc: *const ffi::rtx_scene_desc, width: u32, height: u32, samples: usize, seed: u64) -> Result<Vec<u8>, RtxError> {
        let bytes = width as usize * height as usize * 16;
        let mut pixels = vec![0u8; width as usize * height as usize * 4];
        unsafe {
            let mut scene = ptr::null_mut();
            check(ffi::rtx_scene_create(self.ctx, desc, &mut scene))?;
            let mut accum: *mut c_void = ptr::null_mut();
            let result = (|| {
                check(ffi::rtx_malloc(self.ctx, bytes, &mut accum))?;
                check(ffi::rtx_memset_zero(self.ctx, accum, bytes))?;
                // rtx_render takes at most 2^24 samples per pixel per call: a frame is rendered in chunks of sample indices
                let mut begin = 0usize;
                while begin < samples {
                    let count = (samples - begin).min(1 << 20);
                    let params = ffi::rtx_render_params { width: width as i32, height: height as i32, spp_begin: begin as i32,
                                                          spp_count: count as i32, max_depth: 50, _pad: 0, seed };
                    check(ffi::rtx_render(self.ctx, scene, &params, accum as *mut f32, ptr::null_mut()))?;
                    begin += count;
                }
                check(ffi::rtx_tonemap_rgba8(self.ctx, accum as *const f32, width as i32, height as i32, pixels.as_mut_ptr(), 0))
            })();
            if !accum.is_null() {
                ffi::rtx_free(self.ctx, accum);
            }
            ffi::rtx_scene_destroy(scene);
            result?;
        }
        Ok(pixels)
    }

    /// `render_desc` with adaptive sampling (`rtx_render_adaptive`): every 8x4 tile stops once its noise estimate is
    /// below `adaptive.threshold`, after at least `adaptive.min_spp` and at most `max_spp` samples per pixel.
    pub fn render_adaptive_desc(&self, desc: *const ffi::rtx_scene_desc, width: u32, height: u32, max_spp: usize,
                                adaptive: ffi::rtx_adaptive_params, seed: u64) -> Result<(Vec<u8>, ffi::rtx_adaptive_stats), RtxError> {
        let bytes = width as usize * height as usize * 16;
        let mut pixels = vec![0u8; width as usize * height as usize * 4];
        let mut stats = ffi::rtx_adaptive_stats::default();
        unsafe {
            let mut scene = ptr::null_mut();
            check(ffi::rtx_scene_create(self.ctx, desc, &mut scene))?;
            let mut accum: *mut c_void = ptr::null_mut();
            let mut aux: *mut c_void = ptr::null_mut();
            let result = (|| {
                check(ffi::rtx_malloc(self.ctx, bytes, &mut accum))?;
                check(ffi::rtx_malloc(self.ctx, bytes, &mut aux))?;
                let params = ffi::rtx_render_params { width: width as i32, height: height as i32, spp_begin: 0,
                                                      spp_count: max_spp as i32, max_depth: 50, _pad: 0, seed };
                check(ffi::rtx_render_adaptive(self.ctx, scene, &params, &adaptive, accum as *mut f32, aux as *mut f32, &mut stats))?;
                check(ffi::rtx_tonemap_rgba8(self.ctx, accum as *const f32, width as i32, height as i32, pixels.as_mut_ptr(), 0))
            })();
            for p in [accum, aux] {
                if !p.is_null() {
                    ffi::rtx_free(self.ctx, p);
                }
            }
            ffi::rtx_scene_destroy(scene);
            result?;
        }
        Ok((pixels, stats))
    }
}

impl Drop for Gpu {
    fn drop(&mut self) {
        unsafe { ffi::rtx_ctx_destroy(self.ctx) };
    }
}
