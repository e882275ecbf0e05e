//! `rayrs_lib::gpu` — the B200 backend behind rayrs-lib's scene / material / render API.
//!
//! Drop this file into `rayrs-lib/src/gpu.rs`, apply the four additive patches of `rust/patches/` (a `pub mod gpu;`
//! line and three `pub(crate)` read-only views: `Hittable::flatten`, `Material::flat` / `Emission::flat`,
//! `Bvh::cursor`), link `librayrs_b200.so` (see `rust/build.rs`), and replace the rayon tile loop of
//! `rayrs/src/main.rs:57-101` by
//!
//! ```ignore
//! let image = rayrs_lib::gpu::render_gpu(&c, &s, spp, 50);
//! ```
//!
//! Nothing of the existing API changes: scenes are still built with `Object::sphere`, `Scene::new`, `Camera::new`,
//! the BVH is still the reference's (`Bvh::build`, bvh.rs:199-210).  This module only READS those structures —
//! it is a child of the crate root, so the private fields of `Camera`, `Scene` and `Object` (lib.rs:57-66,216-220,
//! 303-305) are visible to it; the fields private to geometry.rs / material.rs / bvh.rs come through the three
//! views — flattens them into the plain arrays of `include/rayrs_b200.h`, and calls the library.
//!
//! Written against the C header, not compiled in the repository that ships it (there is no Rust toolchain in
//! that image); `examples/render_c.c` is the same algorithm in C and IS compiled and tested there
//! (tests/test_c_example.py: its arrays equal the C++ host mirror's byte for byte).
#![allow(non_camel_case_types)]

use std::ffi::CStr;
use std::os::raw::{c_char, c_int, c_void};
use std::ptr;

use crate::bvh::BvhCursor;
use crate::geometry::{AxisAlignedBoundingBox, FlatGeom};
use crate::image::Image;
use crate::material::FlatMaterial;
use crate::vecmath::{Unit, Vec3, VecElements};
use crate::{Camera, Object, Scene};

// ---------------------------------------------------------------------------------------------------------------
// include/rayrs_b200.h, transcribed (ABI version 2)
// ---------------------------------------------------------------------------------------------------------------
pub const RRS_ABI_VERSION: u32 = 2;
pub const RRS_REF_LEAF: u32 = 0x8000_0000;
pub const RRS_REF_EMPTY: u32 = 0xFFFF_FFFF;
/// RrsRenderParams.flags: next-event estimation of the environment map with MIS (include/rayrs_b200.h)
pub const RRS_FLAG_ENV_SAMPLING: u32 = 64;

#[repr(C)]
#[derive(Clone, Copy, Default)]
pub struct RrsPrim {
    pub type_: u32, // 0 sphere, 1 plane, 2 triangle
    pub obj_id: u32,
    pub material: u32,
    pub emission: i32, // -1 = Emission::Dark
    pub v: [f64; 9],
}

#[repr(C)]
#[derive(Clone, Copy, Default, PartialEq)]
pub struct RrsMaterial {
    pub tag: u32,          // declaration order of `enum Material`, material.rs:57-68
    pub fresnel_kind: u32, // 0 SchlickDielectric, 1 SchlickMetallic
    pub color: [f64; 3],
    pub spec_color: [f64; 3],
    pub alpha: f64,
    pub ior: f64,
}

#[repr(C)]
#[derive(Clone, Copy, Default, PartialEq)]
pub struct RrsEmission {
    pub strength: f64,
    pub color: [f64; 3],
}

#[repr(C)]
#[derive(Clone, Copy)]
pub struct RrsNode {
    pub lo0: [f32; 3],
    pub hi0: [f32; 3],
    pub lo1: [f32; 3],
    pub hi1: [f32; 3],
    pub ref0: u32,
    pub ref1: u32,
    pub flags: u32,
    pub pad: u32,
}

#[repr(C)]
#[derive(Clone, Copy)]
pub struct RrsNodeF64 {
    pub lo0: [f64; 3],
    pub hi0: [f64; 3],
    pub lo1: [f64; 3],
    pub hi1: [f64; 3],
    pub ref0: u32,
    pub ref1: u32,
    pub flags: u32,
    pub pad: [u32; 5],
}

#[repr(C)]
pub struct RrsSceneDesc {
    pub abi_version: u32,
    pub n_prims: u32,
    pub prims: *const RrsPrim,
    pub n_nodes: u32,
    pub nodes: *const RrsNode,
    pub nodes_f64: *const RrsNodeF64,
    pub max_depth: u32,
    pub n_materials: u32,
    pub materials: *const RrsMaterial,
    pub n_emissions: u32,
    pub emissions: *const RrsEmission,
    pub hdri_width: u32,
    pub hdri_height: u32,
    pub hdri_rgb: *const f32,
    pub t_min: f64,
    pub t_max: f64,
    pub flags: u32,
    pub refill_lanes: u32,
}

#[repr(C)]
#[derive(Clone, Copy, Default)]
pub struct RrsCamera {
    pub origin: [f64; 3],
    pub e_x: [f64; 3],
    pub e_y: [f64; 3],
    pub z_scaled: [f64; 3],
    pub width: f64,
    pub height: f64,
    pub ppc: u32,
    pub x_pixels: u32,
    pub y_pixels: u32,
}

#[repr(C)]
#[derive(Clone, Copy, Default)]
pub struct RrsRenderParams {
    pub width: u32,
    pub height: u32,
    pub spp: u32,
    pub sample_offset: u32,
    pub spp_total: u32,
    pub max_bounces: u32,
    pub seed: u64,
    pub queue_capacity: u32,
    pub flags: u32,
}

#[repr(C)]
#[derive(Clone, Copy, Default, Debug)]
pub struct RrsStats {
    pub rays: u64,
    pub paths: u64,
    pub kernel_launches: u64,
    pub iterations: u64,
    pub nan_pixels: u64,
    pub negative_pixels: u64,
    pub device_ms: f64,
    pub extend_ms: f64,
    pub shade_ms: f64,
    pub generate_ms: f64,
    pub nodes_visited: u64,
    pub prims_tested: u64,
    pub kernel_form: u64,
    pub census_mismatch_pixels: u64,
}

#[repr(C)]
pub struct RrsScene {
    _private: [u8; 0],
}
#[repr(C)]
pub struct RrsComm {
    _private: [u8; 0],
}

#[link(name = "rayrs_b200")]
extern "C" {
    fn rrs_scene_create(desc: *const RrsSceneDesc, device: c_int, out: *mut *mut RrsScene) -> c_int;
    fn rrs_scene_create_multi(desc: *const RrsSceneDesc, devices: *const c_int, n: c_int, out: *mut *mut RrsScene) -> c_int;
    fn rrs_scene_destroy(scene: *mut RrsScene);
    fn rrs_render(scene: *mut RrsScene, camera: *const RrsCamera, params: *const RrsRenderParams, out_rgb: *mut f32) -> c_int;
    fn rrs_comm_init_all(devices: *const c_int, n: c_int, out: *mut *mut RrsComm) -> c_int;
    fn rrs_comm_destroy(comm: *mut RrsComm);
    fn rrs_render_multi(
        scenes: *const *mut RrsScene,
        n_local: c_int,
        comm: *mut RrsComm,
        camera: *const RrsCamera,
        params: *const RrsRenderParams,
        out_rgb: *mut f32,
        out_is_device: c_int,
        cuda_streams: *const *mut c_void,
    ) -> c_int;
    fn rrs_stats(scene: *mut RrsScene, out: *mut RrsStats) -> c_int;
    // parity probes of the environment sampler (RRS_FLAG_ENV_SAMPLING)
    #[allow(dead_code)]
    fn rrs_env_sample(scene: *mut RrsScene, u: *const f64, n: usize, dir_pdf: *mut f64) -> c_int;
    #[allow(dead_code)]
    fn rrs_env_pdf(scene: *mut RrsScene, dirs: *const f64, n: usize, pdf: *mut f64) -> c_int;
    fn rrs_last_error() -> *const c_char;
    fn rrs_device_count() -> c_int;
}

/// The reference's error convention is panic-on-bad-input (`assert!`) and no `Result` on the render path
/// (SURVEY.md 8b): a non-zero status becomes a panic carrying the library's message.
fn check(status: c_int, what: &str) {
    if status != 0 {
        let msg = unsafe { CStr::from_ptr(rrs_last_error()) }.to_string_lossy().into_owned();
        panic!("{} failed with status {}: {}", what, status, msg);
    }
}

// ---------------------------------------------------------------------------------------------------------------
// Flattening: Scene -> the arrays of RrsSceneDesc
// ---------------------------------------------------------------------------------------------------------------
/// Largest f32 that is <= x / smallest f32 that is >= x: fp32 boxes are rounded OUTWARD from the reference's
/// f64 boxes so that the fp32 slab test never rejects what the f64 test accepts.
fn round_down(x: f64) -> f32 {
    let f = x as f32; // round to nearest
    if (f as f64) > x { next_after(f, false) } else { f }
}
fn round_up(x: f64) -> f32 {
    let f = x as f32;
    if (f as f64) < x { next_after(f, true) } else { f }
}
fn next_after(f: f32, up: bool) -> f32 {
    if f.is_nan() || f.is_infinite() {
        return f;
    }
    if f == 0.0 {
        let tiny = f32::from_bits(1);
        return if up { tiny } else { -tiny };
    }
    let bits = f.to_bits();
    // moving away from zero increments the magnitude bits, towards zero decrements them
    let away = (f > 0.0) == up;
    f32::from_bits(if away { bits + 1 } else { bits - 1 })
}

fn xyz(v: Vec3) -> [f64; 3] {
    [v.x(), v.y(), v.z()]
}
fn uxyz(v: Unit<Vec3>) -> [f64; 3] {
    [v.x(), v.y(), v.z()] // VecElements for Unit<Vector<T>>, vecmath.rs:466
}
fn box_lo(b: &AxisAlignedBoundingBox) -> [f64; 3] {
    [b.xmin(), b.ymin(), b.zmin()]
}
fn box_hi(b: &AxisAlignedBoundingBox) -> [f64; 3] {
    [b.xmax(), b.ymax(), b.zmax()]
}
/// A box with zero extent on an axis can never pass `AxisAlignedBoundingBox::intersect` (geometry.rs:474,491,508:
/// `tmax <= tmin` on that axis): the reference never enters such a `Node`, so everything below it is unreachable.
fn degenerate(b: &AxisAlignedBoundingBox) -> bool {
    !(b.xmax() > b.xmin() && b.ymax() > b.ymin() && b.zmax() > b.zmin())
}

const EMPTY_LO: [f32; 3] = [f32::INFINITY; 3];
const EMPTY_HI: [f32; 3] = [f32::NEG_INFINITY; 3];

fn empty_node() -> (RrsNode, RrsNodeF64) {
    (
        RrsNode { lo0: EMPTY_LO, hi0: EMPTY_HI, lo1: EMPTY_LO, hi1: EMPTY_HI, ref0: RRS_REF_EMPTY, ref1: RRS_REF_EMPTY, flags: 0, pad: 0 },
        RrsNodeF64 {
            lo0: [f64::INFINITY; 3],
            hi0: [f64::NEG_INFINITY; 3],
            lo1: [f64::INFINITY; 3],
            hi1: [f64::NEG_INFINITY; 3],
            ref0: RRS_REF_EMPTY,
            ref1: RRS_REF_EMPTY,
            flags: 0,
            pad: [0; 5],
        },
    )
}

fn make_leaf(first: u32, count: u32) -> u32 {
    RRS_REF_LEAF | ((count - 1) << 28) | first
}

/// What a parent stores about one child: the reference, whether the child is a bare `LeafNode` (no box of its own
/// in the reference), the reference's exact box and the box the fp32 traversal culls with.
struct ChildSlot {
    reference: u32,
    bare: bool,
    exact: Option<([f64; 3], [f64; 3])>,
    cull: Option<([f64; 3], [f64; 3])>,
}

#[derive(Default)]
pub struct FlatScene {
    pub prims: Vec<RrsPrim>,
    pub nodes: Vec<RrsNode>,
    pub nodes_f64: Vec<RrsNodeF64>,
    pub materials: Vec<RrsMaterial>,
    pub emissions: Vec<RrsEmission>,
    pub hdri_rgb: Vec<f32>,
    pub hdri_width: u32,
    pub hdri_height: u32,
    pub max_depth: u32,
    pub dead_nodes: u32,
    pub t_min: f64,
    pub t_max: f64,
}

impl FlatScene {
    /// `Scene` -> flat arrays.  The walk is the reference's own DFS (children left to right, bvh.rs:391-415), so the
    /// order in which primitives are appended IS the tie-break priority of `RayIntersection::update` (bvh.rs:50-72).
    pub fn from_scene(scene: &Scene) -> FlatScene {
        let mut f = FlatScene::default();
        f.t_min = scene.t_range.start;
        f.t_max = scene.t_range.end;
        // HDRI: f64 RGB -> f32 RGB, row-major, row 0 = top (Image::pixel(i, j) = image[i * width + j], image.rs:183-186)
        let (w, h) = (scene.hdri.width(), scene.hdri.height());
        f.hdri_width = w as u32;
        f.hdri_height = h as u32;
        f.hdri_rgb.reserve(3 * w * h);
        for i in 0..h {
            for j in 0..w {
                let p = scene.hdri.pixel(i, j);
                f.hdri_rgb.extend_from_slice(&[p.x() as f32, p.y() as f32, p.z() as f32]);
            }
        }
        // node 0 = virtual root: child 0 is the reference root with ITS box (the root's own slab test), child 1 empty
        let (n, n64) = empty_node();
        f.nodes.push(n);
        f.nodes_f64.push(n64);
        let root = scene.bvh.cursor();
        let root_box = root.bbox().expect("the root of a Bvh is a Node (bvh.rs:227-316)");
        let slot = f.flatten_child(&root, root_box, 1);
        f.set_child(0, 0, &slot);
        f
    }

    fn material_index(&mut self, m: &FlatMaterial) -> u32 {
        let rec = material_record(m);
        if let Some(i) = self.materials.iter().position(|x| *x == rec) {
            return i as u32;
        }
        self.materials.push(rec);
        (self.materials.len() - 1) as u32
    }

    fn emission_index(&mut self, e: Option<(f64, Vec3)>) -> i32 {
        match e {
            None => -1, // Emission::Dark
            Some((strength, color)) => {
                let rec = RrsEmission { strength, color: xyz(color) };
                if let Some(i) = self.emissions.iter().position(|x| *x == rec) {
                    return i as i32;
                }
                self.emissions.push(rec);
                (self.emissions.len() - 1) as i32
            }
        }
    }

    /// Append one object's primitive record; returns its index (= DFS leaf position).
    fn push_prim(&mut self, obj: &Object) -> u32 {
        let material = self.material_index(&obj.mat.flat());
        let emission = self.emission_index(obj.emission.flat());
        let mut p = RrsPrim { obj_id: self.prims.len() as u32, material, emission, ..RrsPrim::default() };
        match obj.geom.flatten() {
            FlatGeom::Sphere { radius2, origin } => {
                p.type_ = 0;
                p.v[0] = radius2; // Sphere stores radius^2 (geometry.rs:98-101)
                p.v[1] = origin.x();
                p.v[2] = origin.y();
                p.v[3] = origin.z();
            }
            FlatGeom::Plane { axis, umin, umax, vmin, vmax, pos } => {
                p.type_ = 1;
                p.v[0] = axis as u32 as f64; // declaration order of `enum Axis`, geometry.rs:159-167
                p.v[1] = umin;
                p.v[2] = umax;
                p.v[3] = vmin;
                p.v[4] = vmax;
                p.v[5] = pos;
            }
            FlatGeom::Triangle { p1, p2, p3 } => {
                p.type_ = 2;
                p.v[0..3].copy_from_slice(&xyz(p1));
                p.v[3..6].copy_from_slice(&xyz(p2));
                p.v[6..9].copy_from_slice(&xyz(p3));
            }
        }
        self.prims.push(p);
        (self.prims.len() - 1) as u32
    }

    /// Flatten the subtree under `c` (a child of a node whose box is `parent_box`); `depth` = length of the chain of
    /// RrsNodes that ends at the PARENT.  Returns what the parent stores about this child.
    fn flatten_child(&mut self, c: &BvhCursor, parent_box: &AxisAlignedBoundingBox, depth: u32) -> ChildSlot {
        // bare LeafNode: the 1-object side of a split.  The reference tests it whenever the parent is entered (it has
        // no box); cull with the primitive's own box, or with the parent's when that box has no volume (a plane).
        if let Some(obj) = c.object() {
            let first = self.push_prim(obj);
            let own = obj.geom.bbox();
            let cull = if degenerate(&own) { parent_box } else { &own };
            return ChildSlot {
                reference: make_leaf(first, 1),
                bare: true,
                exact: Some((box_lo(&own), box_hi(&own))),
                cull: Some((box_lo(cull), box_hi(cull))),
            };
        }
        let bbox = c.bbox().unwrap();
        let children = c.children();
        if degenerate(bbox) {
            // dead subtree (SURVEY.md F6): its primitives are unreachable in the reference and are not emitted
            self.dead_nodes += 1;
            return ChildSlot { reference: RRS_REF_EMPTY, bare: false, exact: None, cull: None };
        }
        let exact = Some((box_lo(bbox), box_hi(bbox)));
        // leaf group: a Node whose children are all LeafNodes (<= 4 objects, bvh.rs:304-315).  A binary Node always
        // has a Node child (it holds >= 5 objects, so one side holds >= 2).
        if children.iter().all(|ch| ch.object().is_some()) {
            assert!(!children.is_empty() && children.len() <= 4);
            let first = self.prims.len() as u32;
            for ch in &children {
                self.push_prim(ch.object().unwrap());
            }
            return ChildSlot { reference: make_leaf(first, children.len() as u32), bare: false, exact, cull: exact };
        }
        // binary Node -> one RrsNode holding the boxes of BOTH children (pre-order numbering: the left subtree is
        // contiguous behind its parent)
        assert!(children.len() == 2);
        let index = self.nodes.len() as u32;
        let (n, n64) = empty_node();
        self.nodes.push(n);
        self.nodes_f64.push(n64);
        self.max_depth = self.max_depth.max(depth + 1);
        for (k, ch) in children.iter().enumerate() {
            let slot = self.flatten_child(ch, bbox, depth + 1);
            self.set_child(index as usize, k, &slot);
        }
        ChildSlot { reference: index, bare: false, exact, cull: exact }
    }

    fn set_child(&mut self, node: usize, k: usize, s: &ChildSlot) {
        if node == 0 {
            self.max_depth = self.max_depth.max(1);
        }
        let (n, d) = (&mut self.nodes[node], &mut self.nodes_f64[node]);
        if s.bare {
            n.flags |= 1 << k;
            d.flags |= 1 << k;
        }
        let (lo, hi, dlo, dhi) = match (s.cull, s.exact) {
            (Some((clo, chi)), Some((elo, ehi))) => (
                [round_down(clo[0]), round_down(clo[1]), round_down(clo[2])],
                [round_up(chi[0]), round_up(chi[1]), round_up(chi[2])],
                elo,
                ehi,
            ),
            _ => (EMPTY_LO, EMPTY_HI, [f64::INFINITY; 3], [f64::NEG_INFINITY; 3]), // empty child: inverted box
        };
        if k == 0 {
            n.ref0 = s.reference;
            n.lo0 = lo;
            n.hi0 = hi;
            d.ref0 = s.reference;
            d.lo0 = dlo;
            d.hi0 = dhi;
        } else {
            n.ref1 = s.reference;
            n.lo1 = lo;
            n.hi1 = hi;
            d.ref1 = s.reference;
            d.lo1 = dlo;
            d.hi1 = dhi;
        }
    }

    fn desc(&self) -> RrsSceneDesc {
        RrsSceneDesc {
            abi_version: RRS_ABI_VERSION,
            n_prims: self.prims.len() as u32,
            prims: self.prims.as_ptr(),
            n_nodes: self.nodes.len() as u32,
            nodes: self.nodes.as_ptr(),
            nodes_f64: self.nodes_f64.as_ptr(), // lets rrs_intersect(.., precision = 64) verify against the exact boxes
            max_depth: self.max_depth,
            n_materials: self.materials.len() as u32,
            materials: self.materials.as_ptr(),
            n_emissions: self.emissions.len() as u32,
            emissions: if self.emissions.is_empty() { ptr::null() } else { self.emissions.as_ptr() },
            hdri_width: self.hdri_width,
            hdri_height: self.hdri_height,
            hdri_rgb: self.hdri_rgb.as_ptr(),
            t_min: self.t_min,
            t_max: self.t_max,
            flags: 0,
            refill_lanes: 0,
        }
    }
}

/// `enum Material` (material.rs:57-68) -> RrsMaterial.  The constructors' arguments are what the C ABI takes; the
/// structs store `alpha * alpha` (CookTorrance::new, material.rs:703-714), so alpha goes back through a square root
/// (the library squares it again in f64 and rounds to f32: the 1-ulp f64 difference cannot survive).
fn material_record(m: &FlatMaterial) -> RrsMaterial {
    let mut r = RrsMaterial::default();
    match *m {
        FlatMaterial::LambertianDiffuse { color } => {
            r.tag = 0;
            r.color = xyz(color);
        }
        FlatMaterial::Reflect { color } => {
            r.tag = 1;
            r.color = xyz(color);
        }
        FlatMaterial::Refract { color, ior } => {
            r.tag = 2;
            r.color = xyz(color);
            r.ior = ior;
        }
        FlatMaterial::Glass { color, ior } => {
            r.tag = 3;
            r.color = xyz(color);
            r.ior = ior;
        }
        FlatMaterial::CookTorrance { color, alpha2, dielectric_ior, metallic_r0 } => {
            r.tag = 4;
            r.color = xyz(color);
            r.alpha = alpha2.sqrt();
            match (dielectric_ior, metallic_r0) {
                (Some(ior), _) => {
                    r.fresnel_kind = 0;
                    r.ior = ior;
                }
                (None, Some(r0)) => {
                    r.fresnel_kind = 1;
                    r.spec_color = xyz(r0);
                }
                (None, None) => unreachable!(),
            }
        }
        FlatMaterial::CookTorranceRefract { color, alpha2, ior } => {
            r.tag = 5;
            r.color = xyz(color);
            r.alpha = alpha2.sqrt();
            r.ior = ior;
        }
        FlatMaterial::CookTorranceGlass { color, alpha2, ior } => {
            r.tag = 6;
            r.color = xyz(color);
            r.alpha = alpha2.sqrt();
            r.ior = ior;
        }
        FlatMaterial::Plastic { color, spec_color, alpha2, ior } => {
            r.tag = 7;
            r.color = xyz(color); // the diffuse colour
            r.spec_color = xyz(spec_color); // the colour of the inner CookTorrance (Plastic::new, material.rs:880-896)
            r.alpha = alpha2.sqrt();
            r.ior = ior;
        }
        FlatMaterial::NoReflect => r.tag = 8,
    }
    r
}

/// The derived camera fields exactly as `Camera::new` computed them (lib.rs:113-132): the FOV quirk
/// (z scaled by width / tan(fov / 2)) stays on the host.
fn camera_record(c: &Camera) -> RrsCamera {
    RrsCamera {
        origin: xyz(c.origin),
        e_x: uxyz(c.e_x),
        e_y: uxyz(c.e_y),
        z_scaled: xyz(c.z),
        width: c.width,
        height: c.height,
        ppc: c.ppc,
        x_pixels: c.x_pixels() as u32,
        y_pixels: c.y_pixels() as u32,
    }
}

// ---------------------------------------------------------------------------------------------------------------
// The device half of a Scene, and the render call
// ---------------------------------------------------------------------------------------------------------------
/// The scene on one or more GPUs.  Build it once per `Scene` and reuse it across renders (upload is not free);
/// `render_gpu` below builds a temporary one per call, like the reference builds nothing ahead of its tile loop.
pub struct GpuScene {
    handles: Vec<*mut RrsScene>,
    comm: *mut RrsComm,
}

impl GpuScene {
    /// All usable B200s of the box.
    pub fn new(scene: &Scene) -> GpuScene {
        let n = unsafe { rrs_device_count() };
        assert!(n > 0, "no sm_100 device: rayrs_b200 has no CPU fallback");
        GpuScene::on_devices(scene, &(0..n).collect::<Vec<c_int>>())
    }

    pub fn on_devices(scene: &Scene, devices: &[c_int]) -> GpuScene {
        assert!(!devices.is_empty());
        let flat = FlatScene::from_scene(scene); // validated and converted once, uploaded to every device
        let desc = flat.desc();
        let mut handles = vec![ptr::null_mut(); devices.len()];
        let mut comm = ptr::null_mut();
        unsafe {
            if devices.len() == 1 {
                check(rrs_scene_create(&desc, devices[0], handles.as_mut_ptr()), "rrs_scene_create");
            } else {
                check(rrs_scene_create_multi(&desc, devices.as_ptr(), devices.len() as c_int, handles.as_mut_ptr()), "rrs_scene_create_multi");
                check(rrs_comm_init_all(devices.as_ptr(), devices.len() as c_int, &mut comm), "rrs_comm_init_all");
            }
        }
        GpuScene { handles, comm }
    }

    /// The tile loop of rayrs/src/main.rs:57-101: `spp` samples of every pixel, mean radiance per pixel.  With
    /// several GPUs the samples are split inside the one call (one NCCL reduce); the RNG is keyed by the global
    /// sample index, so the image does not depend on the number of GPUs (up to fp32 summation order).
    pub fn render(&self, c: &Camera, spp: u32, max_bounces: u32) -> Image {
        let cam = camera_record(c);
        let (w, h) = (cam.x_pixels as usize, cam.y_pixels as usize);
        let params = RrsRenderParams {
            width: cam.x_pixels,
            height: cam.y_pixels,
            spp,
            sample_offset: 0,
            spp_total: spp,
            max_bounces,
            seed: 0x5EED_B200,
            queue_capacity: 0,
            flags: 0,
        };
        let mut rgb = vec![0f32; 3 * w * h];
        unsafe {
            if self.handles.len() == 1 {
                check(rrs_render(self.handles[0], &cam, &params, rgb.as_mut_ptr()), "rrs_render");
            } else {
                check(
                    rrs_render_multi(self.handles.as_ptr(), self.handles.len() as c_int, self.comm, &cam, &params, rgb.as_mut_ptr(), 0, ptr::null()),
                    "rrs_render_multi",
                );
            }
        }
        // the reference prints these per pixel (main.rs:81-88); the library counts them
        let st = self.stats();
        if st.nan_pixels > 0 {
            println!("NaN in {} pixel(s)", st.nan_pixels);
        }
        if st.negative_pixels > 0 {
            println!("Negative value in {} pixel(s)", st.negative_pixels);
        }
        let pixels: Vec<Vec3> = rgb.chunks_exact(3).map(|p| Vec3::new(p[0] as f64, p[1] as f64, p[2] as f64)).collect();
        Image::from_pixels(w, h, pixels) // image.rs:167-173: row-major, row 0 = top, like Image::from_blocks
    }

    /// Statistics of the last render (device 0 carries the resolve's pixel census).
    pub fn stats(&self) -> RrsStats {
        let mut st = RrsStats::default();
        unsafe { check(rrs_stats(self.handles[0], &mut st), "rrs_stats") };
        st
    }
}

impl Drop for GpuScene {
    fn drop(&mut self) {
        unsafe {
            if !self.comm.is_null() {
                rrs_comm_destroy(self.comm);
            }
            for h in &self.handles {
                rrs_scene_destroy(*h);
            }
        }
    }
}

/// Drop-in for the rayon tile loop of `rayrs/src/main.rs:57-101`.
pub fn render_gpu(c: &Camera, s: &Scene, spp: u32, max_bounces: u32) -> Image {
    GpuScene::new(s).render(c, spp, max_bounces)
}
