"""Python face of the host mirror: the names and argument meanings of rayrs-lib's public API
(Camera, Scene, Object, Material, Fresnel, Emission, BvhHeuristic, render) over the C++ host
library, which in turn drives the CUDA backend through the C ABI.

    reference                                         here
    Camera::new(origin, up, lookat, fov, w, h, ppi)   Camera(origin, up, lookat, fov, w, h, ppi)
    Material::CookTorrance(CookTorrance::new(..))     Material.cook_torrance(color, alpha, Fresnel.schlick_metallic(r0))
    Object::sphere(radius, origin, mat, emission)     Object.sphere(radius, origin, mat, emission)
    Scene::new(objects, z_near, z_far, heuristic, hdri)   Scene(objects, z_near, z_far, heuristic, hdri)
    the tile loop of rayrs/src/main.rs:57-101         render_gpu(camera, scene, spp, max_bounces)

Python only assembles tables of numbers and calls native code; BVH construction, flattening
and rendering are C++/CUDA.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field
from typing import Iterable, Sequence

import numpy as np

from . import _ffi

# material.rs:57-68 declaration order
MAT_LAMBERTIAN, MAT_REFLECT, MAT_REFRACT, MAT_GLASS, MAT_COOK_TORRANCE = 0, 1, 2, 3, 4
MAT_COOK_TORRANCE_REFRACT, MAT_COOK_TORRANCE_GLASS, MAT_PLASTIC, MAT_NO_REFLECT = 5, 6, 7, 8
FRESNEL_DIELECTRIC, FRESNEL_METALLIC = 0, 1


class Axis:
    X, XRev, Y, YRev, Z, ZRev = range(6)


def _v3(v) -> np.ndarray:
    a = np.asarray(v, dtype=np.float64).reshape(3)
    return a


@dataclass(frozen=True)
class Fresnel:
    kind: int
    ior: float = 0.0
    r0: tuple = (0.0, 0.0, 0.0)

    @staticmethod
    def schlick_dielectric(ior: float) -> "Fresnel":
        return Fresnel(FRESNEL_DIELECTRIC, float(ior))

    @staticmethod
    def schlick_metallic(r0) -> "Fresnel":
        return Fresnel(FRESNEL_METALLIC, 0.0, tuple(_v3(r0)))


@dataclass(frozen=True)
class Material:
    """One row of the material table: [tag, color rgb, alpha, ior, fresnel kind, r0/spec rgb, 0, 0]."""
    row: tuple

    @staticmethod
    def _make(tag, color=(0, 0, 0), alpha=0.0, ior=0.0, kind=0, aux=(0, 0, 0)) -> "Material":
        c, a = _v3(color), _v3(aux)
        return Material((float(tag), c[0], c[1], c[2], float(alpha), float(ior), float(kind), a[0], a[1], a[2], 0.0, 0.0))

    @staticmethod
    def lambertian_diffuse(color):
        return Material._make(MAT_LAMBERTIAN, color)

    @staticmethod
    def reflect(color):
        return Material._make(MAT_REFLECT, color)

    @staticmethod
    def refract(color, ior):
        return Material._make(MAT_REFRACT, color, ior=ior)

    @staticmethod
    def glass(color, ior):
        return Material._make(MAT_GLASS, color, ior=ior)

    @staticmethod
    def cook_torrance(color, alpha, fresnel: Fresnel):
        return Material._make(MAT_COOK_TORRANCE, color, alpha, fresnel.ior, fresnel.kind, fresnel.r0)

    @staticmethod
    def cook_torrance_refract(color, alpha, ior):
        return Material._make(MAT_COOK_TORRANCE_REFRACT, color, alpha, ior)

    @staticmethod
    def cook_torrance_glass(color, alpha, ior):
        return Material._make(MAT_COOK_TORRANCE_GLASS, color, alpha, ior)

    @staticmethod
    def plastic(color, spec_color, alpha, ior):
        return Material._make(MAT_PLASTIC, color, alpha, ior, FRESNEL_DIELECTRIC, spec_color)

    @staticmethod
    def no_reflect():
        return Material._make(MAT_NO_REFLECT)


@dataclass(frozen=True)
class Emission:
    strength: float = 0.0
    color: tuple = (0.0, 0.0, 0.0)
    dark: bool = True

    @staticmethod
    def Dark() -> "Emission":
        return Emission()

    @staticmethod
    def new(strength, color) -> "Emission":
        return Emission(float(strength), tuple(_v3(color)), False)


@dataclass
class Object:
    """One object or a batch of objects sharing material and emission.
    rows: n x 12 float64 = [type, 0, 0, payload x 9] — the host table layout (host_capi.cpp) with the material / emission
    index columns left for build_tables to fill, so a mesh goes into the table as one contiguous copy."""
    rows: np.ndarray
    mat: Material
    emission: Emission

    @staticmethod
    def sphere(radius, origin, mat, emission=Emission()):
        o = _v3(origin)
        return Object(np.array([[0, 0, 0, radius, o[0], o[1], o[2], 0, 0, 0, 0, 0]], dtype=np.float64), mat, emission)

    @staticmethod
    def plane(axis, umin, umax, vmin, vmax, pos, mat, emission=Emission()):
        return Object(np.array([[1, 0, 0, axis, umin, umax, vmin, vmax, pos, 0, 0, 0]], dtype=np.float64), mat, emission)

    @staticmethod
    def triangle(p1, p2, p3, mat, emission=Emission()):
        return Object(np.concatenate([[2.0, 0.0, 0.0], _v3(p1), _v3(p2), _v3(p3)])[None, :], mat, emission)

    @staticmethod
    def from_triangles(tris, mat, emission=Emission()):
        """tris: (n, 3, 3) vertex positions, counter-clockwise (lib.rs:407-415)."""
        t = np.asarray(tris, dtype=np.float64).reshape(-1, 9)
        rows = np.empty((t.shape[0], 12))
        rows[:, 0] = 2.0
        rows[:, 1:3] = 0.0
        rows[:, 3:12] = t
        return Object(rows, mat, emission)

    @staticmethod
    def from_spheres(centers, radius, mat, emission=Emission()):
        c = np.asarray(centers, dtype=np.float64).reshape(-1, 3)
        rows = np.zeros((c.shape[0], 12))
        rows[:, 3] = radius
        rows[:, 4:7] = c
        return Object(rows, mat, emission)

    @staticmethod
    def box_geom(lower_left, upper_right, mat, emission=Emission()):
        """lib.rs:438-507 — the same six planes in the same order."""
        ll, ur = _v3(lower_left), _v3(upper_right)
        return [
            Object.plane(Axis.X, ll[1], ur[1], ll[2], ur[2], ll[0], mat, emission),
            Object.plane(Axis.XRev, ll[1], ur[1], ll[2], ur[2], ur[0], mat, emission),
            Object.plane(Axis.ZRev, ll[0], ur[0], ll[1], ur[1], ll[2], mat, emission),
            Object.plane(Axis.Z, ll[0], ur[0], ll[1], ur[1], ur[2], mat, emission),
            Object.plane(Axis.YRev, ll[0], ur[0], ll[2], ur[2], ll[1], mat, emission),
            Object.plane(Axis.Y, ll[0], ur[0], ll[2], ur[2], ll[1], mat, emission),
        ]


@dataclass(frozen=True)
class BvhHeuristic:
    kind: int  # 0 Midpoint, 1 Sah
    splits: int = 0

    @staticmethod
    def Midpoint():
        return BvhHeuristic(0, 0)

    @staticmethod
    def Sah(splits: int):
        return BvhHeuristic(1, int(splits))


@dataclass
class SceneTables:
    """The flat tables that describe a Vec<Object> (host_capi.cpp layout)."""
    objs: np.ndarray  # n x 12
    mats: np.ndarray  # m x 12
    emis: np.ndarray  # k x 4


def build_tables(objects: Iterable[Object]) -> SceneTables:
    mats: list[Material] = []
    emis: list[Emission] = []
    objects = list(objects)
    total = sum(o.rows.shape[0] for o in objects)
    objs = np.empty((total, 12), dtype=np.float64)  # filled slice by slice: no per-object temporaries, no concatenate
    pos = 0
    for o in objects:
        if o.mat not in mats:
            mats.append(o.mat)
        mi = mats.index(o.mat)
        ei = -1
        if not o.emission.dark:
            if o.emission not in emis:
                emis.append(o.emission)
            ei = emis.index(o.emission)
        n = o.rows.shape[0]
        rows = objs[pos:pos + n]
        rows[...] = o.rows
        rows[:, 1] = mi
        rows[:, 2] = ei
        pos += n
    m = np.array([mm.row for mm in mats], dtype=np.float64).reshape(-1, 12)
    e = np.array([[em.strength, *em.color] for em in emis], dtype=np.float64).reshape(-1, 4)
    return SceneTables(objs, np.ascontiguousarray(m), np.ascontiguousarray(e))


class Image:
    """image.rs Image: width, height, row-major pixels (row 0 = top)."""

    def __init__(self, width: int, height: int, pixels: np.ndarray):
        self.width, self.height = int(width), int(height)
        self.pixels = np.ascontiguousarray(np.asarray(pixels, dtype=np.float64).reshape(self.height, self.width, 3))

    @staticmethod
    def from_pixels(width, height, pixels):
        return Image(width, height, pixels)


class Camera:
    """Camera::new lib.rs:99-133.  Raises like the reference panics."""

    def __init__(self, origin, up, lookat, fov, width, height, ppi):
        lib = _ffi.host_lib()
        self.c = _ffi.RrsCamera()
        o, u, l = _v3(origin), _v3(up), _v3(lookat)
        rc = lib.rrh_camera_new(o.ctypes.data, u.ctypes.data, l.ctypes.data, float(fov), float(width), float(height),
                                int(ppi), C.byref(self.c))
        if rc != 0:
            raise ValueError(lib.rrh_last_error().decode())
        self.params = dict(origin=o, up=u, lookat=l, fov=float(fov), width=float(width), height=float(height), ppi=int(ppi))

    def x_pixels(self) -> int:
        return int(self.c.x_pixels)

    def y_pixels(self) -> int:
        return int(self.c.y_pixels)

    def derived17(self) -> np.ndarray:
        """origin, e_x, e_y, z_scaled, width, height, ppc, x_pixels, y_pixels as 17 doubles."""
        c = self.c
        return np.array([*c.origin, *c.e_x, *c.e_y, *c.z_scaled, c.width, c.height, c.ppc, c.x_pixels, c.y_pixels],
                        dtype=np.float64)


class Scene:
    """Scene::new lib.rs:227-245: builds the reference BVH on the host (C++), flattens it and
    uploads it to GPU `device`.  upload=False builds the host half only (no GPU needed)."""

    def __init__(self, objects: Sequence[Object], z_near: float, z_far: float, heuristic: BvhHeuristic, hdri: Image,
                 device: int = 0, with_f64: bool = True, upload: bool = True, devices: Sequence[int] | None = None,
                 scene_flags: int = 0, refill_lanes: int = 0, bvh_threads: int = 0, device_build: bool = False,
                 topology: bool = True):
        """devices: the GPUs that hold the scene (default [device]); the BVH is built and flattened once and
        uploaded to each, and render_gpu() then splits the samples over them (rrs_render_multi).
        scene_flags / refill_lanes: RrsSceneDesc.flags / .refill_lanes (measurement switches).
        device_build: build the reference tree on the GPU (rrs_bvh_build, the same tree) instead of on the host.
        topology: keep the oracle-format dump of the tree (flat()[3:5]); tests need it, a renderer does not."""
        lib = _ffi.host_lib()
        flat = []
        for o in objects:
            flat.extend(o if isinstance(o, (list, tuple)) else [o])
        self.tables = build_tables(flat)
        self.hdri = hdri
        self.z_near, self.z_far, self.heuristic = float(z_near), float(z_far), heuristic
        t = self.tables
        h = np.ascontiguousarray(hdri.pixels, dtype=np.float64)
        self.devices = [int(d) for d in devices] if devices else [int(device)]
        devs = (C.c_int * len(self.devices))(*self.devices)
        self._p = lib.rrh_scene_new(t.objs.ctypes.data, t.objs.shape[0], t.mats.ctypes.data, t.mats.shape[0],
                                    t.emis.ctypes.data if t.emis.size else None, t.emis.shape[0], heuristic.kind,
                                    heuristic.splits, h.ctypes.data, hdri.width, hdri.height, float(z_near),
                                    float(z_far), int(device), int(with_f64), int(upload), int(scene_flags),
                                    int(refill_lanes), int(bvh_threads), devs, len(self.devices), int(device_build), int(topology))
        if not self._p:
            raise ValueError(lib.rrh_last_error().decode())
        info = (C.c_uint64 * 7)()
        bs = C.c_double()
        lib.rrh_scene_info(self._p, info, C.byref(bs))
        self.n_nodes, self.n_prims, self.max_depth, self.dead_nodes, self.n_materials, self._topo_len, self._n_boxes = (
            int(x) for x in info)
        self.build_seconds = bs.value
        t7 = (C.c_double * 7)()
        lib.rrh_scene_build_timing(self._p, t7)
        self.build_timing = dict(zip(("boxes", "tree", "numbering", "flatten", "depth", "topology", "tree_device"), (float(x) for x in t7)))
        self.handle = lib.rrh_scene_handle(self._p) if upload else None
        self.handles = [lib.rrh_scene_handle_at(self._p, i) for i in range(len(self.devices))] if upload else []

    def close(self):
        if getattr(self, "_p", None):
            _ffi.host_lib().rrh_scene_free(self._p)
            self._p = None
            self.handle = None
            self.handles = []

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- host-side views (CPU only) ----------------------------------------------------
    def flat(self):
        """(nodes, nodes_f64, prim_order, topology, boxes, prims) copies of the flattened BVH."""
        lib = _ffi.host_lib()
        nodes = (_ffi.RrsNode * self.n_nodes)()
        nodes64 = (_ffi.RrsNodeF64 * self.n_nodes)()
        order = np.zeros(self.n_prims, dtype=np.uint32)
        topo = np.zeros(self._topo_len, dtype=np.int64)
        boxes = np.zeros((self._n_boxes, 6), dtype=np.float64)
        prims = (_ffi.RrsPrim * self.n_prims)()
        lib.rrh_scene_copy(self._p, nodes, nodes64, order.ctypes.data, topo.ctypes.data, boxes.ctypes.data, prims)
        return nodes, nodes64, order, topo, boxes, prims

    # ---- device-side entry points (C ABI) ----------------------------------------------
    def _need_gpu(self):
        if not self.handle:
            raise _ffi.RayrsError(_ffi.RRS_ERR_NO_DEVICE, "scene has no device half (upload=False)")

    def intersect(self, rays: np.ndarray, precision: int = 32):
        """Bvh::intersect for rays (n x 6: origin, direction) -> (obj_id int32, t float64)."""
        self._need_gpu()
        r = np.ascontiguousarray(rays, dtype=np.float64).reshape(-1, 6)
        ids = np.zeros(r.shape[0], dtype=np.int32)
        t = np.zeros(r.shape[0], dtype=np.float64)
        _ffi.check(_ffi.cuda_lib().rrs_intersect(self.handle, r.ctypes.data, r.shape[0], ids.ctypes.data, t.ctypes.data,
                                                 int(precision)))
        return ids, t

    def material_evaluate(self, material: int, normal_view: np.ndarray, u: np.ndarray, cases_form: bool = False) -> np.ndarray:
        self._need_gpu()
        nv = np.ascontiguousarray(normal_view, dtype=np.float64).reshape(-1, 6)
        uu = np.ascontiguousarray(u, dtype=np.float64).reshape(-1, 3)
        out = np.zeros((nv.shape[0], 7), dtype=np.float32)
        _ffi.check(_ffi.cuda_lib().rrs_material_evaluate(self.handle, int(material) | (0x80000000 if cases_form else 0), nv.ctypes.data, uu.ctypes.data,
                                                         nv.shape[0], out.ctypes.data))
        return out

    def material_evaluate_pdf(self, material: int, light, pos_normal_view: np.ndarray, u: np.ndarray) -> np.ndarray:
        """Material::evaluate(position, normal, view, Some(Pdf::Hittable(light))) — material.rs:91-109,259-281,943-959,1027-1034:
        the reference's dormant next-event-estimation hook.  `light`: the _ffi.RrsPrim record of the sampled primitive
        (an entry of flat()[5]); pos_normal_view n x 9; u n x 4 draws in call order -> n x 7 doubles."""
        self._need_gpu()
        q = np.ascontiguousarray(pos_normal_view, dtype=np.float64).reshape(-1, 9)
        uu = np.ascontiguousarray(u, dtype=np.float64).reshape(-1, 4)
        out = np.zeros((q.shape[0], 7), dtype=np.float64)
        _ffi.check(_ffi.cuda_lib().rrs_material_evaluate_pdf(self.handle, int(material), C.byref(light), q.ctypes.data, uu.ctypes.data,
                                                             q.shape[0], out.ctypes.data))
        return out

    def background(self, dirs: np.ndarray) -> np.ndarray:
        self._need_gpu()
        d = np.ascontiguousarray(dirs, dtype=np.float64).reshape(-1, 3)
        out = np.zeros((d.shape[0], 3), dtype=np.float32)
        _ffi.check(_ffi.cuda_lib().rrs_background(self.handle, d.ctypes.data, d.shape[0], out.ctypes.data))
        return out

    def env_sample(self, u: np.ndarray) -> np.ndarray:
        """rrs_env_sample: n x 2 uniforms in [0, 1) -> n x 4 (unit direction xyz, solid-angle density) as the
        RRS_FLAG_ENV_SAMPLING render draws them."""
        self._need_gpu()
        uu = np.ascontiguousarray(u, dtype=np.float64).reshape(-1, 2)
        out = np.zeros((uu.shape[0], 4), dtype=np.float64)
        _ffi.check(_ffi.cuda_lib().rrs_env_sample(self.handle, uu.ctypes.data, uu.shape[0], out.ctypes.data))
        return out

    def env_pdf(self, dirs: np.ndarray) -> np.ndarray:
        """rrs_env_pdf: the environment sampler's solid-angle density of n directions (n x 3)."""
        self._need_gpu()
        d = np.ascontiguousarray(dirs, dtype=np.float64).reshape(-1, 3)
        out = np.zeros(d.shape[0], dtype=np.float64)
        _ffi.check(_ffi.cuda_lib().rrs_env_pdf(self.handle, d.ctypes.data, d.shape[0], out.ctypes.data))
        return out

    def rng_uniforms(self, seed: int, pixel: int, sample: int, slot: int) -> np.ndarray:
        self._need_gpu()
        out = np.zeros(4, dtype=np.float32)
        _ffi.check(_ffi.cuda_lib().rrs_rng_uniforms(self.handle, seed, pixel, sample, slot, out.ctypes.data))
        return out

    def stats(self, index: int = 0) -> dict:
        """RrsStats of the last render on the index-th device of the scene (waits for an asynchronous render)."""
        self._need_gpu()
        st = _ffi.RrsStats()
        _ffi.check(_ffi.cuda_lib().rrs_stats(self.handles[index], C.byref(st)))
        return {name: getattr(st, name) for name, _ in _ffi.RrsStats._fields_}

    def comm(self) -> int:
        """The scene's own communicator over its devices (single-process multi-GPU)."""
        self._need_gpu()
        c = _ffi.host_lib().rrh_scene_comm(self._p)
        if not c:
            raise _ffi.RayrsError(_ffi.RRS_ERR_COMM, _ffi.host_lib().rrh_last_error().decode())
        return c


DEFAULT_SEED = 0x5EEDB200
# render flag: next-event estimation of the environment map with MIS (include/rayrs_b200.h)
RRS_FLAG_ENV_SAMPLING = _ffi.RRS_FLAG_ENV_SAMPLING


def render_params(camera: Camera, spp: int, max_bounces: int, seed: int = DEFAULT_SEED, sample_offset: int = 0,
                  spp_total: int = 0, queue_capacity: int = 0, flags: int = 0) -> _ffi.RrsRenderParams:
    return _ffi.RrsRenderParams(camera.x_pixels(), camera.y_pixels(), int(spp), int(sample_offset), int(spp_total),
                                int(max_bounces), int(seed), int(queue_capacity), int(flags))


def render_gpu(camera: Camera, scene: Scene, spp: int, max_bounces: int = 50, out: np.ndarray | None = None,
               **opts) -> np.ndarray:
    """Drop-in for the tile loop of rayrs/src/main.rs:57-101: H x W x 3 float32 mean radiance
    (host buffer; host<->device copies inside the call).  max_bounces defaults to the
    reference's literal 50 (main.rs:77)."""
    scene._need_gpu()
    p = render_params(camera, spp, max_bounces, **opts)
    if out is None:
        out = np.empty((camera.y_pixels(), camera.x_pixels(), 3), dtype=np.float32)
    if len(scene.handles) > 1:  # the scene lives on several GPUs: still one call
        render_multi(camera, scene.handles, scene.comm(), spp, max_bounces, out_ptr=out.ctypes.data, **opts)
        return out
    _ffi.check(_ffi.cuda_lib().rrs_render(scene.handle, C.byref(camera.c), C.byref(p), out.ctypes.data))
    return out


def sample_range(rank: int, world: int, spp: int) -> tuple[int, int]:
    """rrs_sample_range: (first global sample, number of samples) of `rank`."""
    first, count = C.c_uint32(), C.c_uint32()
    _ffi.check(_ffi.cuda_lib().rrs_sample_range(int(rank), int(world), int(spp), C.byref(first), C.byref(count)))
    return int(first.value), int(count.value)


class Comm:
    """RrsComm of one process per GPU (torchrun): rank 0 makes the id, `exchange(bytes) -> bytes` hands it to
    the other ranks (e.g. a torch.distributed broadcast — plumbing), every rank joins."""

    def __init__(self, world: int, rank: int, device: int, exchange):
        lib = _ffi.cuda_lib()
        uid = _ffi.RrsUniqueId()
        if rank == 0:
            _ffi.check(lib.rrs_comm_unique_id(C.byref(uid)))
        raw = exchange(bytes(uid) if rank == 0 else None)
        C.memmove(C.byref(uid), raw, 128)
        self.ptr = C.c_void_p()
        _ffi.check(lib.rrs_comm_init_rank(C.byref(uid), int(world), int(rank), int(device), C.byref(self.ptr)))
        self.world, self.rank = world, rank

    def close(self):
        if self.ptr:
            _ffi.cuda_lib().rrs_comm_destroy(self.ptr)
            self.ptr = None


def render_multi(camera: Camera, handles, comm, spp: int, max_bounces: int = 50, out_ptr: int = 0, out_is_device: bool = False,
                 streams=None, **opts) -> None:
    """rrs_render_multi: `spp` TOTAL samples split over the ranks of `comm`, one NCCL reduce, mean image written on
    global rank 0 to out_ptr (host memory, or rank 0's GPU when out_is_device).  handles: this process's scene
    handles, one per local device of the communicator; comm: RrsComm pointer (Scene.comm() or Comm.ptr)."""
    p = render_params(camera, spp, max_bounces, **opts)
    hs = (C.c_void_p * len(handles))(*handles)
    st = (C.c_void_p * len(handles))(*streams) if streams is not None else None
    _ffi.check(_ffi.cuda_lib().rrs_render_multi(hs, len(handles), comm, C.byref(camera.c), C.byref(p), C.c_void_p(out_ptr),
                                                int(out_is_device), st))


def render_accumulate(camera: Camera, scene: Scene, spp: int, max_bounces: int, d_sum_ptr: int, stream_ptr: int = 0,
                      **opts) -> None:
    """Accumulate this call's samples into a DEVICE float4-per-pixel buffer (multi-GPU path)."""
    scene._need_gpu()
    p = render_params(camera, spp, max_bounces, **opts)
    _ffi.check(_ffi.cuda_lib().rrs_render_accumulate(scene.handle, C.byref(camera.c), C.byref(p), C.c_void_p(d_sum_ptr),
                                                     C.c_void_p(stream_ptr)))


def resolve(scene: Scene, d_sum_ptr: int, width: int, height: int, spp_total: int, out_ptr: int, out_is_device: bool,
            stream_ptr: int = 0) -> None:
    scene._need_gpu()
    _ffi.check(_ffi.cuda_lib().rrs_resolve(scene.handle, C.c_void_p(d_sum_ptr), width, height, spp_total,
                                           C.c_void_p(out_ptr), int(out_is_device), C.c_void_p(stream_ptr)))


def to_raw_bytes(scene: Scene, d_sum_ptr: int, width: int, height: int, spp_total: int, gamma: float = 1.0 / 2.2,
                 out_ptr: int = 0, stream_ptr: int = 0):
    """Image::to_raw_bytes (image.rs:193-222) on the device, fused with the division by spp.  With out_ptr == 0
    returns (H x W x 3 uint8 host array, {clamped, nan, negative} pixel counts); otherwise writes the bytes to the
    DEVICE buffer at out_ptr and returns (None, counts)."""
    scene._need_gpu()
    census = (C.c_uint64 * 3)()
    host = None
    if out_ptr == 0:
        host = np.empty((height, width, 3), dtype=np.uint8)
        ptr, on_device = host.ctypes.data, 0
    else:
        ptr, on_device = out_ptr, 1
    _ffi.check(_ffi.cuda_lib().rrs_to_raw_bytes(scene.handle, C.c_void_p(d_sum_ptr), width, height, spp_total, float(gamma),
                                                C.c_void_p(ptr), on_device, C.c_void_p(stream_ptr), census))
    return host, {"clamped": int(census[0]), "nan": int(census[1]), "negative": int(census[2])}
