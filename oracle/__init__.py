"""ctypes wrapper of the CPU oracle (oracle/oracle.cpp).

TEST INFRASTRUCTURE ONLY.  Importable from tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs; the product package rayrs_b200 never imports it.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from pathlib import Path

import numpy as np

_DIR = Path(__file__).resolve().parent
LIB_PATH = _DIR / "liboracle.so"
_lib = None


def build(force: bool = False) -> Path:
    src = _DIR / "oracle.cpp"
    if force or not LIB_PATH.exists() or LIB_PATH.stat().st_mtime < src.stat().st_mtime:
        subprocess.run(["make", "-C", str(_DIR)] + (["-B"] if force else []), check=True, stdout=subprocess.PIPE,
                       stderr=subprocess.STDOUT)
    return LIB_PATH


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        if not LIB_PATH.exists():
            build()
        L = C.CDLL(str(LIB_PATH))
        vp, u64, u32, i32, dbl = C.c_void_p, C.c_uint64, C.c_uint32, C.c_int, C.c_double
        L.orc_scene_create.restype = vp
        L.orc_scene_create.argtypes = [vp, u64, vp, u64, vp, u64, i32, u32, i32, vp, u64, u64, dbl, dbl]
        L.orc_scene_destroy.argtypes = [vp]
        L.orc_tree_dump.restype = u64
        L.orc_tree_dump.argtypes = [vp, vp, u64, vp, u64]
        L.orc_intersect.argtypes = [vp, vp, u64, vp, vp, i32]
        L.orc_intersect_stable.argtypes = [vp, vp, u64, dbl, dbl, vp, i32]
        L.orc_intersect_sensitivity.argtypes = [vp, vp, u64, dbl, dbl, vp, vp, i32]
        L.orc_camera_new.argtypes = [vp, vp, vp, dbl, dbl, dbl, u32, vp]
        L.orc_primary_rays.argtypes = [vp, u32, u32, vp, vp, vp, u64, u64, i32, vp]
        L.orc_render.argtypes = [vp, vp, u32, u32, u32, u32, u32, u64, i32, i32, vp, vp]
        L.orc_render_env.restype = i32
        L.orc_render_env.argtypes = [vp, vp, u32, u32, u32, u32, u32, u64, i32, i32, vp, vp]
        L.orc_env_table.restype = i32
        L.orc_env_table.argtypes = [vp, vp, vp, vp]
        L.orc_env_sample.restype = i32
        L.orc_env_sample.argtypes = [vp, vp, u64, vp]
        L.orc_env_pdf.restype = i32
        L.orc_env_pdf.argtypes = [vp, vp, u64, vp]
        L.orc_material_evaluate.argtypes = [vp, vp, vp, u64, vp]
        L.orc_material_evaluate_pdf.argtypes = [vp, vp, vp, vp, u64, vp]
        L.orc_hittable_area_sample.argtypes = [vp, vp, vp]
        L.orc_background.argtypes = [vp, vp, u64, vp]
        L.orc_sphere_intersect.restype = i32
        L.orc_sphere_intersect.argtypes = [dbl, vp, vp, vp]
        L.orc_plane_intersect.restype = i32
        L.orc_plane_intersect.argtypes = [i32, dbl, dbl, dbl, dbl, dbl, vp, vp]
        L.orc_triangle_intersect.restype = i32
        L.orc_triangle_intersect.argtypes = [vp, vp, vp, vp]
        L.orc_aabb_intersect.restype = i32
        L.orc_aabb_intersect.argtypes = [vp, vp, dbl, dbl]
        L.orc_scene_bbox.argtypes = [vp, vp]
        L.orc_orthonormal_basis.argtypes = [vp, vp]
        L.orc_vecmath_ops.argtypes = [vp, vp, dbl, vp]
        L.orc_philox.argtypes = [vp, vp, vp, i32]
        L.orc_rng_uniforms.argtypes = [u64, u32, u32, u32, i32, vp]
        L.orc_traversal_counts.argtypes = [vp, vp, u64, vp, vp, vp]
        L.orc_collect_path_rays.restype = u64
        L.orc_collect_path_rays.argtypes = [vp, vp, u32, u32, u32, u32, u64, i32, u32, vp, u64]
        L.orc_hardware_threads.restype = i32
        _lib = L
    return _lib


def _d(a):
    return np.ascontiguousarray(a, dtype=np.float64)


RNG_WIDE, RNG_MATCHED = 0, 1  # 53-bit uniforms / the 24-bit values the GPU backend draws


def hardware_threads() -> int:
    return int(lib().orc_hardware_threads()) or (os.cpu_count() or 1)


class OracleScene:
    """Scene::new on the CPU restatement.  `tables` is rayrs_b200.api.SceneTables (plain arrays)."""

    def __init__(self, tables, hdri_pixels: np.ndarray, z_near=1e-6, z_far=1e6, heuristic=(1, 1000), build_mode=0):
        self.objs, self.mats, self.emis = _d(tables.objs), _d(tables.mats), _d(tables.emis)
        h = _d(hdri_pixels)
        self.hdri = h
        hh, hw = h.shape[0], h.shape[1]
        self._p = lib().orc_scene_create(self.objs.ctypes.data, self.objs.shape[0], self.mats.ctypes.data,
                                         self.mats.shape[0], self.emis.ctypes.data if self.emis.size else None,
                                         self.emis.shape[0], int(heuristic[0]), int(heuristic[1]), int(build_mode),
                                         h.ctypes.data, hw, hh, float(z_near), float(z_far))

    def close(self):
        if self._p:
            lib().orc_scene_destroy(self._p)
            self._p = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def tree_dump(self):
        n = lib().orc_tree_dump(self._p, None, 0, None, 0)
        topo = np.zeros(n, dtype=np.int64)
        n_nodes = int((topo.size))  # upper bound for boxes
        boxes = np.zeros((n_nodes, 6), dtype=np.float64)
        lib().orc_tree_dump(self._p, topo.ctypes.data, n, boxes.ctypes.data, boxes.size)
        nn = int((topo < 0).sum())
        return topo, boxes[:nn]

    def intersect(self, rays, nthreads=0):
        r = _d(rays).reshape(-1, 6)
        ids = np.zeros(r.shape[0], dtype=np.int32)
        t = np.zeros(r.shape[0], dtype=np.float64)
        lib().orc_intersect(self._p, r.ctypes.data, r.shape[0], ids.ctypes.data, t.ctypes.data,
                            nthreads or hardware_threads())
        return ids, t

    def intersect_stable(self, rays, eps_dir=2e-6, eps_org=2e-5, nthreads=0):
        r = _d(rays).reshape(-1, 6)
        st = np.zeros(r.shape[0], dtype=np.uint8)
        lib().orc_intersect_stable(self._p, r.ctypes.data, r.shape[0], eps_dir, eps_org, st.ctypes.data,
                                   nthreads or hardware_threads())
        return st.astype(bool)

    def intersect_sensitivity(self, rays, eps_dir=2e-6, eps_org=2e-5, nthreads=0):
        """(stable, tchange): the stability probe plus the largest relative change of t over its 12 perturbed
        rays — how well conditioned t is with respect to the ray (0 where not stable or a miss)."""
        r = _d(rays).reshape(-1, 6)
        st = np.zeros(r.shape[0], dtype=np.uint8)
        tc = np.zeros(r.shape[0], dtype=np.float64)
        lib().orc_intersect_sensitivity(self._p, r.ctypes.data, r.shape[0], eps_dir, eps_org, st.ctypes.data,
                                        tc.ctypes.data, nthreads or hardware_threads())
        return st.astype(bool), tc

    def render(self, cam17, W, H, spp, max_bounces=50, seed=0x5EEDB200, sample_offset=0, rng_mode=RNG_MATCHED, nthreads=0,
               env=False):
        """env=True: with the GPU backend's environment sampling (RRS_FLAG_ENV_SAMPLING); the stats then also hold
        shadow_rays (counted in rays as well).  Raises ValueError for a map the flag refuses (non-finite texels)."""
        out = np.zeros((H, W, 3), dtype=np.float64)
        stats = np.zeros(8, dtype=np.uint64)
        c = _d(cam17)
        args = (self._p, c.ctypes.data, W, H, spp, sample_offset, max_bounces, seed, rng_mode,
                nthreads or hardware_threads(), out.ctypes.data, stats.ctypes.data)
        if env:
            if lib().orc_render_env(*args) != 0:
                raise ValueError("the environment map cannot be tabulated for sampling (non-finite texels)")
        else:
            lib().orc_render(*args)
        st = dict(rays=int(stats[0]), scatters=int(stats[1]), nan_pixels=int(stats[2]),
                  negative_pixels=int(stats[3]), seconds=float(stats[4]) * 1e-6,
                  reentry_total=int(stats[5]), reentry_lost=int(stats[6]))
        if env:
            st["shadow_rays"] = int(stats[7])
        return out, st

    def env_table(self):
        """The environment-sampling table (rayrs_b200/csrc/api.cu build_env_table): dict(marg (ch,), cond (ch, cw),
        row (ch, 2)) as float32, None for a black map; ValueError for a map with non-finite texels."""
        hh, hw = self.hdri.shape[:2]
        marg = np.zeros(hh - 1, dtype=np.float32)
        cond = np.zeros((hh - 1, hw - 1), dtype=np.float32)
        row = np.zeros((hh - 1, 2), dtype=np.float32)
        rc = lib().orc_env_table(self._p, marg.ctypes.data, cond.ctypes.data, row.ctypes.data)
        if rc < 0:
            raise ValueError("the environment map cannot be tabulated for sampling (non-finite texels)")
        return dict(marg=marg, cond=cond, row=row) if rc == 1 else None

    def env_sample(self, u):
        """rrs_env_sample's inputs (n x 2 uniforms in [0, 1)) -> n x 6: direction xyz, density of the drawn cell,
        cell row, cell column."""
        uu = _d(u).reshape(-1, 2)
        out = np.zeros((uu.shape[0], 6))
        if lib().orc_env_sample(self._p, uu.ctypes.data, uu.shape[0], out.ctypes.data) != 0:
            raise ValueError("nothing to sample: the map is black or has non-finite texels")
        return out

    def env_pdf(self, dirs):
        """rrs_env_pdf: the density of n directions (n x 3) in the cell Scene::background reads them from."""
        d = _d(dirs).reshape(-1, 3)
        out = np.zeros(d.shape[0])
        if lib().orc_env_pdf(self._p, d.ctypes.data, d.shape[0], out.ctypes.data) != 0:
            raise ValueError("the environment map cannot be tabulated for sampling (non-finite texels)")
        return out

    def background(self, dirs):
        d = _d(dirs).reshape(-1, 3)
        out = np.zeros_like(d)
        lib().orc_background(self._p, d.ctypes.data, d.shape[0], out.ctypes.data)
        return out

    def bbox(self):
        out = np.zeros(11)
        lib().orc_scene_bbox(self._p, out.ctypes.data)
        return out

    def traversal_counts(self, rays):
        r = _d(rays).reshape(-1, 6)
        b, h = C.c_uint64(), C.c_uint64()
        p = (C.c_uint64 * 3)()
        lib().orc_traversal_counts(self._p, r.ctypes.data, r.shape[0], C.byref(b), p, C.byref(h))
        return b.value, [int(x) for x in p], h.value  # boxes tested, [spheres, planes, triangles] tested, hits

    def collect_path_rays(self, cam17, W, H, spp, max_bounces, seed=0x5EEDB200, rng_mode=RNG_MATCHED, pixel_stride=1,
                          cap=1 << 20):
        out = np.zeros((cap, 6), dtype=np.float64)
        c = _d(cam17)
        n = lib().orc_collect_path_rays(self._p, c.ctypes.data, W, H, spp, max_bounces, seed, rng_mode, pixel_stride,
                                        out.ctypes.data, cap)
        return out[:n]


def camera_new(origin, up, lookat, fov, width, height, ppi) -> np.ndarray:
    out = np.zeros(17)
    o, u, l = _d(origin), _d(up), _d(lookat)
    lib().orc_camera_new(o.ctypes.data, u.ctypes.data, l.ctypes.data, fov, width, height, ppi, out.ctypes.data)
    return out


def primary_rays(cam17, W, H, rows, cols, samples, seed=0x5EEDB200, rng_mode=RNG_MATCHED) -> np.ndarray:
    rows = np.ascontiguousarray(rows, dtype=np.uint32)
    cols = np.ascontiguousarray(cols, dtype=np.uint32)
    samples = np.ascontiguousarray(samples, dtype=np.uint32)
    out = np.zeros((rows.size, 6))
    c = _d(cam17)
    lib().orc_primary_rays(c.ctypes.data, W, H, rows.ctypes.data, cols.ctypes.data, samples.ctypes.data, rows.size,
                           seed, rng_mode, out.ctypes.data)
    return out


def material_evaluate(mat_row, normal_view, u) -> np.ndarray:
    m, nv, uu = _d(mat_row), _d(normal_view).reshape(-1, 6), _d(u).reshape(-1, 3)
    out = np.zeros((nv.shape[0], 7))
    lib().orc_material_evaluate(m.ctypes.data, nv.ctypes.data, uu.ctypes.data, nv.shape[0], out.ctypes.data)
    return out


def material_evaluate_pdf(mat_row, obj_row, pos_normal_view, u) -> np.ndarray:
    """Material::evaluate with pdf = Some(Pdf::Hittable(geometry of obj_row)) — material.rs:91-109,259-281,943-959,1027-1034.
    obj_row: 12 doubles as the scene tables carry them; pos_normal_view: n x 9; u: n x 4 draws in call order."""
    m, g, q, uu = _d(mat_row), _d(obj_row), _d(pos_normal_view).reshape(-1, 9), _d(u).reshape(-1, 4)
    out = np.zeros((q.shape[0], 7))
    lib().orc_material_evaluate_pdf(m.ctypes.data, g.ctypes.data, q.ctypes.data, uu.ctypes.data, q.shape[0], out.ctypes.data)
    return out


def hittable_area_sample(obj_row, u2):
    """(Hittable::area, Hittable::sample with the two draws u2) of one object row — geometry.rs:138-152,284-299,381-387"""
    g, uu = _d(obj_row), _d(u2)
    out = np.zeros(4)
    lib().orc_hittable_area_sample(g.ctypes.data, uu.ctypes.data, out.ctypes.data)
    return float(out[0]), out[1:].copy()


def sphere_intersect(radius, origin, ray6):
    t = C.c_double()
    o, r = _d(origin), _d(ray6)
    hit = lib().orc_sphere_intersect(radius, o.ctypes.data, r.ctypes.data, C.byref(t))
    return (t.value if hit else None)


def plane_intersect(axis, umin, umax, vmin, vmax, pos, ray6):
    t = C.c_double()
    r = _d(ray6)
    hit = lib().orc_plane_intersect(axis, umin, umax, vmin, vmax, pos, r.ctypes.data, C.byref(t))
    return (t.value if hit else None)


def triangle_intersect(p9, ray6):
    t = C.c_double()
    n = np.zeros(3)
    p, r = _d(p9), _d(ray6)
    hit = lib().orc_triangle_intersect(p.ctypes.data, r.ctypes.data, C.byref(t), n.ctypes.data)
    return (t.value if hit else None), n


def aabb_intersect(box6, ray6, tmin, tmax) -> bool:
    b, r = _d(box6), _d(ray6)
    return bool(lib().orc_aabb_intersect(b.ctypes.data, r.ctypes.data, tmin, tmax))


def vecmath_ops(a, b, s) -> dict:
    """the oracle's Vec3 operators on (a, b, s): add, sub, mul, scalar_mul (s * a), mul_scalar (a * s), dot, cross, mag2 (of a)"""
    out = np.zeros(20)
    aa, bb = _d(a), _d(b)
    lib().orc_vecmath_ops(aa.ctypes.data, bb.ctypes.data, float(s), out.ctypes.data)
    return {"add": out[0:3], "sub": out[3:6], "mul": out[6:9], "scalar_mul": out[9:12], "mul_scalar": out[12:15],
            "dot": float(out[15]), "cross": out[16:19], "mag2": float(out[19])}


def orthonormal_basis(n3):
    out = np.zeros(6)
    n = _d(n3)
    lib().orc_orthonormal_basis(n.ctypes.data, out.ctypes.data)
    return out[:3], out[3:]


def philox(ctr4, key2, rounds: int = 0) -> np.ndarray:
    """Philox4x32 with `rounds` rounds (0 = the render stream's round count, 7)."""
    c = np.ascontiguousarray(ctr4, dtype=np.uint32)
    k = np.ascontiguousarray(key2, dtype=np.uint32)
    out = np.zeros(4, dtype=np.uint32)
    lib().orc_philox(c.ctypes.data, k.ctypes.data, out.ctypes.data, int(rounds))
    return out


def rng_uniforms(seed, pixel, sample, slot, mode=RNG_MATCHED) -> np.ndarray:
    out = np.zeros(4)
    lib().orc_rng_uniforms(seed, pixel, sample, slot, mode, out.ctypes.data)
    return out


def to_raw_bytes(image: np.ndarray, gamma: float = 1.0 / 2.2):
    """Image::to_raw_bytes, rayrs-lib/src/image.rs:193-222, restated in numpy f64: per pixel the three censuses
    the reference prints (clamped > 1, NaN, negative), then clip(0, 1) (min then max, both dropping NaN like
    f64::min/max, vecmath.rs:389-397), powf(gamma), and (255.99 * x) as u8 (Rust's saturating float cast).
    Returns (H x W x 3 uint8, {clamped, nan, negative})."""
    v = np.asarray(image, dtype=np.float64)
    nan = np.isnan(v).any(axis=-1)
    with np.errstate(invalid="ignore"):
        neg = (v < 0.0).any(axis=-1)
        bright = (v > 1.0).any(axis=-1)
        c = np.fmax(np.fmin(v, 1.0), 0.0)
        q = 255.99 * np.power(c, gamma)
    out = np.clip(np.nan_to_num(q, nan=0.0), 0.0, 255.0).astype(np.uint8)  # truncation toward zero
    return out, {"clamped": int(bright.sum()), "nan": int(nan.sum()), "negative": int(neg.sum())}
