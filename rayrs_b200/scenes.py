"""Scene descriptions: the reference's test scenes (rayrs-lib/src/test_scenes.rs) with a
configurable film size, plus the synthetic inputs the reference does not ship (HDRI, meshes;
its *.hdr / *.obj / *.ply are git-ignored) — SURVEY.md 8(d).

Every builder returns a SceneSpec (camera arguments + object list + heuristic); `spec.scene()`
turns it into a GPU `Scene`, and tests hand `spec.tables()` to the CPU oracle, so both sides
consume identical numbers.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Callable

import numpy as np

from .api import Axis, BvhHeuristic, Camera, Emission, Fresnel, Image, Material, Object, Scene, build_tables

Z_NEAR, Z_FAR = 0.000_001, 1_000_000.0  # rayrs/src/main.rs:52
PPI = 100  # -> ppc = round(100 * 2.54) = 254 pixels per cm


def film(width_px: int, height_px: int):
    """Film size in cm such that Camera::x_pixels()/y_pixels() == (width_px, height_px) at PPI."""
    return width_px / 254.0, height_px / 254.0


@dataclass
class SceneSpec:
    name: str
    camera_args: dict
    objects: list
    heuristic: BvhHeuristic
    max_bounces: int = 50  # rayrs/src/main.rs:77

    def camera(self) -> Camera:
        return Camera(**self.camera_args)

    def tables(self):
        flat = []
        for o in self.objects:
            flat.extend(o if isinstance(o, (list, tuple)) else [o])
        return build_tables(flat)

    def scene(self, hdri: Image, device: int = 0, **kw) -> Scene:
        return Scene(self.objects, Z_NEAR, Z_FAR, self.heuristic, hdri, device=device, **kw)


# ---------------------------------------------------------------------------------------
# synthetic environment (closed form, no RNG): vertical gradient + Gaussian sun + ground tint,
# clipped to [0, 3] as rayrs/src/main.rs:43 clips the decoded HDR
# ---------------------------------------------------------------------------------------
def synthetic_hdri(width: int = 2048, height: int = 1024) -> Image:
    i = np.arange(height, dtype=np.float64)[:, None]
    j = np.arange(width, dtype=np.float64)[None, :]
    theta = np.pi * i / (height - 1)          # 0 at the top row (dir.y = +1), lib.rs:259-264
    phi = 2.0 * np.pi * j / (width - 1)       # phi = atan2(z, x) + pi
    cy = np.cos(theta)
    sy = np.sin(theta)
    dx, dz = -np.cos(phi) * sy, -np.sin(phi) * sy
    dy = cy + 0.0 * phi
    up = np.clip(dy, 0.0, 1.0)
    zenith = np.array([0.35, 0.55, 1.0])
    horizon = np.array([1.0, 0.95, 0.9])
    ground = np.array([0.25, 0.22, 0.2])
    w = np.sqrt(up)[..., None]
    sky = 1.2 * (horizon * (1.0 - w) + zenith * w)
    gnd = ground * (0.5 + 0.5 * np.abs(dy))[..., None]
    img = np.where((dy >= 0.0)[..., None], sky, gnd)
    ts, ps = 0.9, 2.2
    sun = np.array([-np.cos(ps) * np.sin(ts), np.cos(ts), -np.sin(ps) * np.sin(ts)])
    cosang = np.clip(dx * sun[0] + dy * sun[1] + dz * sun[2], -1.0, 1.0)
    ang = np.arccos(cosang)
    img = img + (30.0 * np.exp(-0.5 * (ang / 0.08) ** 2))[..., None] * np.array([1.0, 0.9, 0.75])
    return Image(width, height, np.clip(img, 0.0, 3.0))


def sun_hdri(width: int = 128, height: int = 64, sky: float = 1.0, sun: float = 2000.0) -> Image:
    """Unclipped environment for environment sampling (RRS_FLAG_ENV_SAMPLING): a uniform sky and a 3 x 3-texel sun
    `sun / sky` times brighter, high in the sky — most of the light in a small part of the map."""
    px = np.full((height, width, 3), float(sky))
    px[height // 4 - 1:height // 4 + 2, width // 3 - 1:width // 3 + 2] = (sun, 0.95 * sun, 0.85 * sun)
    return Image(width, height, px)


# ---------------------------------------------------------------------------------------
# test_scenes.rs
# ---------------------------------------------------------------------------------------
def _floor() -> Object:
    # test_scenes.rs:15-21 — rough-metal Cook-Torrance plane (SURVEY.md F4)
    mat = Material.cook_torrance((1.0, 1.0, 1.0), 0.5, Fresnel.schlick_metallic((0.8, 0.8, 0.8)))
    return Object.plane(Axis.Y, -25.0, 25.0, -25.0, 25.0, 0.0, mat, Emission.Dark())


def _single_sphere(name: str, mat: Material, width_px: int, height_px: int) -> SceneSpec:
    # test_scenes.rs:14-44
    w, h = film(width_px, height_px)
    objects = [_floor(), Object.sphere(1.0, (0.0, 1.0, 0.0), mat, Emission.Dark())]
    cam = dict(origin=(0.0, 5.0, 10.0), up=(0.0, 1.0, 0.0), lookat=(0.0, 1.0, 0.0), fov=50.0, width=w, height=h, ppi=PPI)
    return SceneSpec(name, cam, objects, BvhHeuristic.Sah(1000))


def copper_single_sphere(width_px=975, height_px=549):
    # test_scenes.rs:46-53
    return _single_sphere("copper_single_sphere",
                          Material.cook_torrance((1, 1, 1), 0.05, Fresnel.schlick_metallic((0.722, 0.451, 0.2))),
                          width_px, height_px)


def glass_single_sphere(width_px=975, height_px=549):
    # test_scenes.rs:55-58
    return _single_sphere("glass_single_sphere", Material.glass((0.8, 0.8, 0.8), 1.45), width_px, height_px)


def diffuse_single_sphere(width_px=975, height_px=549):
    # test_scenes.rs:60-63
    return _single_sphere("diffuse_single_sphere", Material.lambertian_diffuse((0.8, 0.8, 0.8)), width_px, height_px)


def cook_torrance_glass_single_sphere(width_px=975, height_px=549):
    # test_scenes.rs:65-68
    return _single_sphere("cook_torrance_glass_single_sphere", Material.cook_torrance_glass((0.8, 0.8, 0.8), 0.05, 1.45),
                          width_px, height_px)


def _multiple_spheres(name: str, mats: list, width_px: int, height_px: int, extra: list | None = None,
                      camera: dict | None = None) -> SceneSpec:
    # test_scenes.rs:163-211
    w, h = film(width_px, height_px)
    n = len(mats)
    objects = [_floor()]
    for i, m in enumerate(mats):
        objects.append(Object.sphere(1.0, (2.2 * (i - n // 2), 1.0, 0.0), m, Emission.Dark()))
    if extra:
        objects.extend(extra)
    cam = dict(origin=(0.0, 10.0, 20.0), up=(0.0, 1.0, 0.0), lookat=(0.0, 1.0, 0.0), fov=72.0, width=w, height=h, ppi=PPI)
    if camera:
        cam.update(camera)
    return SceneSpec(name, cam, objects, BvhHeuristic.Sah(1000))


def cook_torrance_spheres_metallic(width_px=1221, height_px=254):
    # test_scenes.rs:213-224
    mats = [Material.cook_torrance((1, 1, 1), 0.01 * (4 * i + 1), Fresnel.schlick_metallic((0.8, 0.8, 0.8))) for i in range(7)]
    return _multiple_spheres("cook_torrance_spheres_metallic", mats, width_px, height_px)


def cook_torrance_spheres_plastic(width_px=1221, height_px=254):
    # test_scenes.rs:226-239
    mats = [Material.plastic((0.8, 0.8, 0.8), (1, 1, 1), 0.01 * (4 * i + 1), 1.45) for i in range(7)]
    return _multiple_spheres("cook_torrance_spheres_plastic", mats, width_px, height_px)


def cook_torrance_spheres_frosted_glass(width_px=1221, height_px=254):
    # test_scenes.rs:241-256
    mats = [Material.cook_torrance_glass((1, 1, 1), 0.01 * (4 * i + 1), 1.45) for i in range(7)]
    return _multiple_spheres("cook_torrance_spheres_frosted_glass", mats, width_px, height_px)


def cook_torrance_spheres_cook_torrance_refract(width_px=1221, height_px=254):
    # test_scenes.rs:258-274
    mats = [Material.cook_torrance_refract((1, 1, 1), 0.01 * (4 * i + 1), 1.45) for i in range(6)]
    mats.insert(0, Material.refract((1, 1, 1), 1.45))
    return _multiple_spheres("cook_torrance_spheres_cook_torrance_refract", mats, width_px, height_px)


def material_test(width_px=1221, height_px=159):
    # test_scenes.rs:276-331
    mats = [
        Material.lambertian_diffuse((0.8, 0.8, 0.8)),
        Material.plastic((0.8, 0.8, 0.8), (1, 1, 1), 0.05, 1.45),
        Material.reflect((0.8, 0.8, 0.8)),
        Material.cook_torrance((1, 1, 1), 0.05, Fresnel.schlick_metallic((0.8, 0.8, 0.8))),
        Material.glass((1, 1, 1), 1.45),
        Material.cook_torrance_glass((1, 1, 1), 0.05, 1.45),
        Material.no_reflect(),
    ]
    return _multiple_spheres("material_test", mats, width_px, height_px,
                             camera=dict(origin=(0.0, 3.0, 20.0), fov=90.0))


# ---------------------------------------------------------------------------------------
# synthetic mesh: closed-form displaced torus (no poles => no zero-area triangles; tilted so
# that no facet is axis aligned => no zero-extent leaf boxes, SURVEY.md F6)
# ---------------------------------------------------------------------------------------
def torus_mesh(nu: int, nv: int, center=(0.0, 1.7, 0.0), major=1.1, minor=0.45, tilt=(0.37, 0.21)):
    """(vertices float32 (nu*nv, 3), faces int32 (2*nu*nv, 3)); 2*nu*nv triangles, CCW outward."""
    u = (np.arange(nu, dtype=np.float64) * (2.0 * np.pi / nu))[:, None]
    v = (np.arange(nv, dtype=np.float64) * (2.0 * np.pi / nv))[None, :]
    r = minor * (1.0 + 0.13 * np.sin(9.0 * u) * np.sin(7.0 * v))
    x = (major + r * np.cos(v)) * np.cos(u)
    z = (major + r * np.cos(v)) * np.sin(u)
    y = r * np.sin(v) + 0.0 * u
    p = np.stack([x, y, z], axis=-1).reshape(-1, 3)
    ax, az = tilt
    rx = np.array([[1, 0, 0], [0, np.cos(ax), -np.sin(ax)], [0, np.sin(ax), np.cos(ax)]])
    rz = np.array([[np.cos(az), -np.sin(az), 0], [np.sin(az), np.cos(az), 0], [0, 0, 1]])
    p = p @ (rz @ rx).T + np.asarray(center, dtype=np.float64)
    iu = np.arange(nu)[:, None]
    iv = np.arange(nv)[None, :]
    a = (iu * nv + iv).ravel()
    b = (((iu + 1) % nu) * nv + iv).ravel()
    c = (((iu + 1) % nu) * nv + (iv + 1) % nv).ravel()
    d = (iu * nv + (iv + 1) % nv).ravel()
    faces = np.concatenate([np.stack([a, d, c], axis=1), np.stack([a, c, b], axis=1)], axis=0).astype(np.int32)
    return p.astype(np.float32), faces


def mesh_triangles(vertices: np.ndarray, faces: np.ndarray) -> np.ndarray:
    """(n, 3, 3) float64 triangle soup from an indexed mesh (what wavefront_obj.rs:15-44 builds)."""
    return vertices.astype(np.float64)[faces]


def mesh_via_ply(vertices: np.ndarray, faces: np.ndarray, tag: str) -> np.ndarray:
    """The BASELINE mesh configurations name a PLY mesh: write the synthetic mesh as binary-LE PLY
    (float32 xyz, uchar-count int32 faces) and read it back through the host PLY loader — the path a
    rayrs user's mesh takes (file -> load_ply_file -> Object::from_triangles)."""
    import tempfile
    from pathlib import Path
    from . import mesh
    # a private directory per call: a fixed shared one would belong to whichever user created it first
    with tempfile.TemporaryDirectory(prefix="rayrs_b200_mesh_") as d:
        path = Path(d) / f"{tag}.ply"
        mesh.write_ply(path, vertices, faces)
        return mesh.load_ply_file(path)


COPPER = dict(color=(1, 1, 1), alpha=0.05, r0=(0.722, 0.451, 0.2))  # test_scenes.rs:154-159


def copper_torus(nu=1000, nv=500, width_px=1920, height_px=1080, heuristic: BvhHeuristic | None = None) -> SceneSpec:
    """obj_scene template (test_scenes.rs:70-109) with the copper material (:154-159) and the
    synthetic torus in place of the unshipped models/suzanne.obj."""
    w, h = film(width_px, height_px)
    mat = Material.cook_torrance(COPPER["color"], COPPER["alpha"], Fresnel.schlick_metallic(COPPER["r0"]))
    verts, faces = torus_mesh(nu, nv)
    objects = [_floor(), Object.from_triangles(mesh_via_ply(verts, faces, f"torus_{nu}x{nv}"), mat, Emission.Dark())]
    cam = dict(origin=(0.0, 5.0, 10.0), up=(0.0, 1.0, 0.0), lookat=(0.0, 1.0, 0.0), fov=50.0, width=w, height=h, ppi=PPI)
    return SceneSpec(f"copper_torus_{2 * nu * nv}", cam, objects, heuristic or BvhHeuristic.Sah(1000))


def glass_torus(nu=200, nv=100, width_px=1920, height_px=1080, heuristic: BvhHeuristic | None = None) -> SceneSpec:
    """glass_suzanne (test_scenes.rs:164-167): the obj_scene template with Glass(1, 1.45) on the mesh — refraction
    through a closed triangle mesh (rays spawned on a triangle, travelling inside, leaving through another)."""
    w, h = film(width_px, height_px)
    mat = Material.glass((1, 1, 1), 1.45)
    verts, faces = torus_mesh(nu, nv)
    objects = [_floor(), Object.from_triangles(mesh_via_ply(verts, faces, f"torus_{nu}x{nv}_glass"), mat, Emission.Dark())]
    cam = dict(origin=(0.0, 5.0, 10.0), up=(0.0, 1.0, 0.0), lookat=(0.0, 1.0, 0.0), fov=50.0, width=w, height=h, ppi=PPI)
    return SceneSpec(f"glass_torus_{2 * nu * nv}", cam, objects, heuristic or BvhHeuristic.Sah(1000))


def emissive_room(width_px=240, height_px=160) -> SceneSpec:
    """Not a reference scene (every shipped one is Emission::Dark, SURVEY.md F11): an emissive sphere and an emissive
    panel light a Lambertian sphere, a plastic sphere and a box (Object::box_geom: planes on all six axis variants)
    standing on the usual floor — exercises Emission::Emissive gathering (lib.rs:533-547, only in the Scatter arm)."""
    w, h = film(width_px, height_px)
    white = Material.lambertian_diffuse((0.8, 0.8, 0.8))
    objects = [
        _floor(),
        Object.sphere(0.6, (-2.4, 0.6, 0.0), white, Emission.new(6.0, (1.0, 0.7, 0.4))),
        Object.sphere(1.0, (0.0, 1.0, 0.0), white),
        Object.sphere(0.8, (2.2, 0.8, 0.4), Material.plastic((0.2, 0.5, 0.8), (1, 1, 1), 0.1, 1.45)),
        Object.plane(Axis.YRev, -1.5, 1.5, -1.5, 1.5, 4.0, Material.lambertian_diffuse((0.5, 0.5, 0.5)), Emission.new(3.0, (0.6, 0.8, 1.0))),
    ] + Object.box_geom((-1.0, 0.0, 1.6), (-0.2, 0.9, 2.4), Material.cook_torrance((1, 1, 1), 0.2, Fresnel.schlick_metallic((0.9, 0.6, 0.3))))
    cam = dict(origin=(0.0, 3.0, 9.0), up=(0.0, 1.0, 0.0), lookat=(0.0, 1.0, 0.0), fov=50.0, width=w, height=h, ppi=PPI)
    return SceneSpec("emissive_room", cam, objects, BvhHeuristic.Sah(1000))


def mixed_scene(nu=2000, nv=1000, width_px=3840, height_px=2160, heuristic: BvhHeuristic | None = None) -> SceneSpec:
    """Config 5: the seven spheres of multiple_spheres (test_scenes.rs:178-189) with the in-scope
    materials of material_test (:276-289), a synthetic torus behind the row, and the floor."""
    mats = [
        Material.lambertian_diffuse((0.8, 0.8, 0.8)),
        Material.plastic((0.8, 0.8, 0.8), (1, 1, 1), 0.05, 1.45),
        Material.cook_torrance((1, 1, 1), 0.05, Fresnel.schlick_metallic((0.8, 0.8, 0.8))),
        Material.glass((1, 1, 1), 1.45),
        Material.cook_torrance_glass((1, 1, 1), 0.05, 1.45),
        Material.cook_torrance(COPPER["color"], COPPER["alpha"], Fresnel.schlick_metallic(COPPER["r0"])),
        Material.cook_torrance_glass((1, 1, 1), 0.25, 1.45),
    ]
    copper = Material.cook_torrance(COPPER["color"], COPPER["alpha"], Fresnel.schlick_metallic(COPPER["r0"]))
    verts, faces = torus_mesh(nu, nv, center=(0.0, 1.7, -4.0))
    extra = [Object.from_triangles(mesh_via_ply(verts, faces, f"torus_{nu}x{nv}_back"), copper, Emission.Dark())]
    spec = _multiple_spheres(f"mixed_{2 * nu * nv}", mats, width_px, height_px, extra=extra)
    if heuristic:
        spec.heuristic = heuristic
    return spec


# ---------------------------------------------------------------------------------------
# BASELINE.json configs
# ---------------------------------------------------------------------------------------
@dataclass
class Config:
    key: str
    description: str
    specs: Callable[[], list]  # list of SceneSpec rendered back to back
    width: int
    height: int
    spp: int
    max_bounces: int


def sun_spheres(width_px=64, height_px=48) -> SceneSpec:
    """A Lambertian and a rough metallic Cook-Torrance sphere (alpha 0.3) on the rough metallic floor, for sun_hdri."""
    w, h = film(width_px, height_px)
    objects = [_floor(),
               Object.sphere(1.0, (-1.2, 1.0, 0.0), Material.lambertian_diffuse((0.8, 0.7, 0.6)), Emission.Dark()),
               Object.sphere(1.0, (1.2, 1.0, 0.0), Material.cook_torrance((0.9, 0.9, 0.9), 0.3, Fresnel.schlick_metallic((0.9, 0.6, 0.3))),
                             Emission.Dark())]
    cam = dict(origin=(0.0, 4.0, 9.0), up=(0.0, 1.0, 0.0), lookat=(0.0, 1.0, 0.0), fov=50.0, width=w, height=h, ppi=PPI)
    return SceneSpec("sun_spheres", cam, objects, BvhHeuristic.Sah(1000), max_bounces=16)


def _c1():
    s = diffuse_single_sphere(512, 512)
    s.max_bounces = 8
    return [s]


CONFIGS = {
    "c1": Config("c1", "diffuse_single_sphere (1 Lambertian sphere + ground), 512x512, 64 spp, max depth 8", _c1, 512, 512, 64, 8),
    "c2": Config("c2", "Cook-Torrance metallic + plastic sphere series (roughness sweep), 1024x1024, 256 spp",
                 lambda: [cook_torrance_spheres_metallic(1024, 1024), cook_torrance_spheres_plastic(1024, 1024)],
                 1024, 1024, 256, 50),
    "c3": Config("c3", "rough + smooth dielectric glass spheres (frosted-glass series + glass sphere), 1920x1080, 512 spp",
                 lambda: [cook_torrance_spheres_frosted_glass(1920, 1080), glass_single_sphere(1920, 1080)],
                 1920, 1080, 512, 50),
    "c4": Config("c4", "synthetic 1M-triangle displaced torus with BVH, copper Cook-Torrance, 1920x1080, 256 spp",
                 lambda: [copper_torus(1000, 500, 1920, 1080)], 1920, 1080, 256, 50),
    "c5": Config("c5", "4K mixed spheres + 4M-triangle synthetic mesh, 3840x2160, 4096 spp, sample-split across GPUs",
                 lambda: [mixed_scene(2000, 1000, 3840, 2160)], 3840, 2160, 4096, 50),
}
