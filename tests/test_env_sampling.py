"""Environment importance sampling with MIS (RRS_FLAG_ENV_SAMPLING).

CPU: a numpy restatement of the sampling table (api.cu build_env_table) and of the sampler / density (env.cuh) —
the density integrates to 1, is positive wherever Scene::background can be non-zero, and the sampler draws
directions with that density (chi^2).
GPU: rrs_env_sample / rrs_env_pdf agree with the restatement; with the flag the render converges to the image
without it (same estimator, Russian roulette and quirks included) on three scenes, with a per-block bound taken
from the measured standard errors of both; the flag lowers the variance on a sun-lit scene; the census holds.
"""
import numpy as np
import pytest
from scipy import stats

from rayrs_b200 import _ffi, api, scenes

G = 1 << 24


# ---------------------------------------------------------------------------------------
# numpy restatement of the table (api.cu build_env_table, quantize_cdf)
# ---------------------------------------------------------------------------------------
def _quantize(w, total):
    k = np.where(w > 0.0, np.maximum(1, np.floor(w / total * G + 0.5)), 0).astype(np.int64)
    big = int(np.argmax(k))
    k[big] += G - int(k.sum())
    assert k[big] >= 1
    start = np.concatenate([[0], np.cumsum(k)[:-1]])
    return (start / G).astype(np.float32)


class EnvTable:
    def __init__(self, pixels):
        px = np.asarray(pixels, dtype=np.float32)
        h, w = px.shape[:2]
        self.w, self.h = w, h
        self.cw, self.ch = w - 1, h - 1
        lum = np.abs(px).max(axis=2)
        m = np.maximum(np.maximum(lum[:-1, :-1], lum[:-1, 1:]), np.maximum(lum[1:, :-1], lum[1:, 1:])).astype(np.float64)
        i = np.arange(self.ch, dtype=np.float64)
        t0, t1 = np.pi * i / self.ch, np.pi * (i + 1) / self.ch
        dcos = 2.0 * np.sin(0.5 * (t0 + t1)) * np.sin(0.5 * (t1 - t0))
        self.cos0 = np.cos(t0).astype(np.float32)
        self.dcos = dcos.astype(np.float32)
        dphi = 2.0 * np.pi / self.cw
        cell = m * dphi * dcos[:, None]
        rows = np.cumsum(cell, axis=1)[:, -1]     # left to right, as the host sums
        total = np.cumsum(rows)[-1]
        assert total > 0
        self.marg = _quantize(rows, total)
        self.cond = np.zeros((self.ch, self.cw), dtype=np.float32)
        for r in range(self.ch):
            if rows[r] > 0:
                self.cond[r] = _quantize(cell[r], rows[r])
        self.pm = np.diff(np.append(self.marg.astype(np.float64), 1.0))
        self.pc = np.diff(np.concatenate([self.cond.astype(np.float64), np.ones((self.ch, 1))], axis=1), axis=1)
        self.inv_dphi = np.float32(self.cw / (2.0 * np.pi))
        # solid-angle density per cell
        self.cell_pdf = self.pm[:, None] * self.pc * float(self.inv_dphi) / self.dcos.astype(np.float64)[:, None]
        self.cell_omega = dphi * dcos[:, None] * np.ones((1, self.cw))

    def coords(self, dirs):
        d = np.asarray(dirs, dtype=np.float64)
        d = d / np.linalg.norm(d, axis=1, keepdims=True)
        phi = np.arctan2(d[:, 2], d[:, 0]) + np.pi
        theta = np.arccos(np.clip(d[:, 1], -1.0, 1.0))
        return phi / (2 * np.pi) * (self.w - 1), theta / np.pi * (self.h - 1)

    def cells(self, dirs):
        x, y = self.coords(dirs)
        j = np.minimum(np.floor(x).astype(np.int64), self.cw - 1)
        i = np.minimum(np.floor(y).astype(np.int64), self.ch - 1)
        return i, j

    def pdf(self, dirs):
        i, j = self.cells(dirs)
        return self.cell_pdf[i, j]

    def sample(self, u):
        """u: n x 2 in [0, 1) -> (dirs n x 3, cell row, cell column, (t0, t1) position inside the cell)."""
        u = np.asarray(u, dtype=np.float64)
        x = np.minimum(np.floor(u * G), G - 1)
        hi, lo = x / G, np.minimum(u * G - x, 1.0)
        i = np.searchsorted(self.marg.astype(np.float64), hi[:, 0], side="right") - 1
        cond = self.cond.astype(np.float64)[i]
        j = np.array([np.searchsorted(c, v, side="right") - 1 for c, v in zip(cond, hi[:, 1])])
        t0 = np.minimum(((hi[:, 0] - self.marg[i]) + lo[:, 0] / G) / self.pm[i], 1.0)
        t1 = np.minimum(((hi[:, 1] - cond[np.arange(len(i)), j]) + lo[:, 1] / G) / self.pc[i, j], 1.0)
        cy = self.cos0[i].astype(np.float64) - t0 * self.dcos[i]
        sy = np.sqrt(np.maximum(0.0, (1 - cy) * (1 + cy)))
        phi = 2 * np.pi * (j + t1) / self.cw
        dirs = np.stack([-sy * np.cos(phi), cy, -sy * np.sin(phi)], axis=1)
        return dirs, i, j, np.stack([t0, t1], axis=1)


def background_np(pixels, dirs):
    """Scene::background (shading.cuh background) in f64."""
    px = np.asarray(pixels, dtype=np.float32).astype(np.float64)
    h, w = px.shape[:2]
    d = np.asarray(dirs, dtype=np.float64)
    d = d / np.linalg.norm(d, axis=1, keepdims=True)
    x = (np.arctan2(d[:, 2], d[:, 0]) + np.pi) / (2 * np.pi) * (w - 1)
    y = np.arccos(np.clip(d[:, 1], -1, 1)) / np.pi * (h - 1)
    xf, yf = np.floor(x), np.floor(y)
    fx, fy = (x - xf)[:, None], (y - yf)[:, None]
    j0 = np.minimum(xf.astype(np.int64), w - 1)
    j1 = np.minimum(j0 + 1, w - 1)
    i0 = np.minimum(yf.astype(np.int64), h - 1)
    i1 = np.minimum(i0 + 1, h - 1)
    return (px[i0, j0] * (1 - fx) * (1 - fy) + px[i1, j0] * (1 - fx) * fy + px[i0, j1] * fx * (1 - fy)
            + px[i1, j1] * fx * fy)


def hot_texel_map(w=16, h=8, at=(3, 11), value=5.0):
    px = np.zeros((h, w, 3))
    px[at[0], at[1]] = (value, 0.5 * value, 0.0)
    return px


def sun_map(w=128, h=64):
    return scenes.sun_hdri(w, h).pixels


def _sphere_grid(n_phi, n_theta):
    """midpoints of a (phi, theta) grid and their solid angles sin(theta) dtheta dphi"""
    phi = (np.arange(n_phi) + 0.5) * 2 * np.pi / n_phi
    th = (np.arange(n_theta) + 0.5) * np.pi / n_theta
    P, T = np.meshgrid(phi, th)
    s = np.sin(T)
    dirs = np.stack([-np.cos(P) * s, np.cos(T), -np.sin(P) * s], axis=-1).reshape(-1, 3)
    return dirs, (s * (2 * np.pi / n_phi) * (np.pi / n_theta)).ravel()


# ---------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("which", ["synthetic", "hot_texel", "sun"])
def test_density_integrates_to_one(which):
    px = {"synthetic": lambda: scenes.synthetic_hdri(128, 64).pixels, "hot_texel": hot_texel_map, "sun": sun_map}[which]()
    t = EnvTable(px)
    # per cell: the CDF steps sum to 1 exactly; the density's fp32 solid-angle factors round to 1e-7
    assert abs((t.cell_pdf * t.cell_omega).sum() - 1.0) < 1e-6
    dirs, dw = _sphere_grid(16 * t.cw, 16 * t.ch)                     # quadrature over the sphere
    assert abs((t.pdf(dirs) * dw).sum() - 1.0) < 1e-4


@pytest.mark.parametrize("which", ["synthetic", "hot_texel", "sun"])
def test_density_positive_where_background_is_not_zero(which):
    px = {"synthetic": lambda: scenes.synthetic_hdri(128, 64).pixels, "hot_texel": hot_texel_map, "sun": sun_map}[which]()
    t = EnvTable(px)
    dirs, _ = _sphere_grid(1000, 1000)
    bg = background_np(px, dirs)
    lit = np.abs(bg).max(axis=1) > 0
    assert lit.any()
    assert np.all(t.pdf(dirs)[lit] > 0)


@pytest.mark.parametrize("which", ["synthetic", "sun"])
def test_sampled_directions_follow_the_density(which):
    px = {"synthetic": lambda: scenes.synthetic_hdri(64, 32).pixels, "sun": lambda: sun_map(64, 32)}[which]()
    t = EnvTable(px)
    rng = np.random.default_rng(7)
    n = 400_000
    dirs, i, j, _ = t.sample(rng.random((n, 2)))
    assert np.allclose(np.linalg.norm(dirs, axis=1), 1, atol=1e-9)
    # the drawn direction lies in the drawn cell (up to the cell boundary)
    x, y = t.coords(dirs)
    assert np.all((x >= j - 1e-6) & (x <= j + 1 + 1e-6) & (y >= i - 1e-6) & (y <= i + 1 + 1e-6))
    # chi^2 over bins of 2 x 2 cells, each split in 2 x 2 sub-cells (the density inside a cell is uniform in solid
    # angle: sub-cell probabilities from the (phi, cos theta) split)
    bi, bj = np.minimum(np.floor(y).astype(int), t.ch - 1), np.minimum(np.floor(x).astype(int), t.cw - 1)
    sub_phi = (x - bj) >= 0.5
    c_mid = np.cos(np.pi * (bi + 0.5) / t.ch)
    sub_th = dirs[:, 1] < c_mid
    key = ((bi // 2) * ((t.cw + 1) // 2) + bj // 2) * 4 + sub_phi * 2 + sub_th
    obs = np.bincount(key, minlength=((t.ch + 1) // 2) * ((t.cw + 1) // 2) * 4).astype(np.float64)
    ii, jj = np.meshgrid(np.arange(t.ch), np.arange(t.cw), indexing="ij")
    p_cell = t.cell_pdf * t.cell_omega
    ct0, ct1, cm = np.cos(np.pi * ii / t.ch), np.cos(np.pi * (ii + 1) / t.ch), np.cos(np.pi * (ii + 0.5) / t.ch)
    frac_upper = (ct0 - cm) / (ct0 - ct1)
    exp = np.zeros_like(obs)
    for sp in (0, 1):
        for sth, fr in ((0, frac_upper), (1, 1 - frac_upper)):
            k = ((ii // 2) * ((t.cw + 1) // 2) + jj // 2) * 4 + sp * 2 + sth
            np.add.at(exp, k.ravel(), (p_cell * 0.5 * fr).ravel() * n)
    keep = exp > 20
    assert obs[~keep].sum() <= max(50, 2 * exp[~keep].sum() + 5 * np.sqrt(exp[~keep].sum() + 1))
    chi2 = float(((obs[keep] - exp[keep]) ** 2 / exp[keep]).sum())
    dof = int(keep.sum()) - 1
    assert stats.chi2.sf(chi2, dof) > 1e-4, (chi2, dof)


def test_flag_is_bound():
    assert _ffi.RRS_FLAG_ENV_SAMPLING == 64
    assert api.RRS_FLAG_ENV_SAMPLING == 64


# ---------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------
def _furnace_spec(W=48, H=48):
    w, h = scenes.film(W, H)
    objects = [api.Object.sphere(1.0, (0.0, 0.0, 0.0), api.Material.lambertian_diffuse((1.0, 1.0, 1.0)), api.Emission.Dark())]
    cam = dict(origin=(0.0, 0.5, 3.0), up=(0.0, 1.0, 0.0), lookat=(0.0, 0.0, 0.0), fov=50.0, width=w, height=h, ppi=scenes.PPI)
    return scenes.SceneSpec("furnace", cam, objects, api.BvhHeuristic.Sah(1000), max_bounces=50)


def _renders(sc, cam, spp, mb, flags, seeds):
    imgs = []
    for s in seeds:
        img = api.render_gpu(cam, sc, spp, mb, seed=s, flags=flags).astype(np.float64)
        st = sc.stats()
        assert st["census_mismatch_pixels"] == 0 and st["nan_pixels"] == 0 and st["negative_pixels"] == 0, st
        imgs.append(img)
    return np.stack(imgs)


def _block_means(imgs, b=8):
    k, H, W, _ = imgs.shape
    Hb, Wb = H // b, W // b
    x = imgs[:, :Hb * b, :Wb * b].sum(axis=3).reshape(k, Hb, b, Wb, b).mean(axis=(2, 4))
    return x.reshape(k, -1)


def assert_same_mean(on, off, alpha=1e-3):
    """Welch test per 8 x 8 block and over the whole image, Bonferroni over the blocks: the bound is set by the
    standard errors measured over independent seeds, not by a tolerance."""
    a, b = _block_means(on), _block_means(off)
    a = np.concatenate([a, a.mean(axis=1, keepdims=True)], axis=1)
    b = np.concatenate([b, b.mean(axis=1, keepdims=True)], axis=1)
    k = a.shape[0]
    ma, mb_ = a.mean(axis=0), b.mean(axis=0)
    va, vb = a.var(axis=0, ddof=1) / k, b.var(axis=0, ddof=1) / k
    se = np.sqrt(va + vb)
    exact = se <= 1e-7 * np.maximum(np.abs(ma), 1e-30)
    assert np.all(np.abs(ma - mb_)[exact] <= 1e-5 * np.abs(mb_[exact]) + 1e-7)
    tcrit = stats.t.isf(alpha / (2 * a.shape[1]), k - 1)
    z = np.abs(ma - mb_)[~exact] / se[~exact]
    worst = float(z.max()) if z.size else 0.0
    assert worst < tcrit, f"block mean differs by {worst:.2f} standard errors (bound {tcrit:.2f})"
    return worst, tcrit


@pytest.fixture(scope="module")
def sun_scene(native_built):
    spec = scenes.sun_spheres()
    sc = spec.scene(scenes.sun_hdri())
    yield spec, sc
    sc.close()


@pytest.mark.gpu
@pytest.mark.parametrize("which", ["synthetic", "sun"])
def test_probes_match_the_restatement(which, native_built):
    px = scenes.synthetic_hdri(256, 128).pixels if which == "synthetic" else sun_map()
    H, W = px.shape[:2]
    sc = scenes.diffuse_single_sphere(32, 32).scene(api.Image(W, H, px))
    t = EnvTable(px)
    rng = np.random.default_rng(3)
    u = rng.random((20000, 2))
    got = sc.env_sample(u)
    dirs, i, j, tt = t.sample(u)
    assert np.max(np.abs(got[:, :3] - dirs)) < 1e-5
    ref = t.cell_pdf[i, j]
    near_edge = np.any((tt < 1e-4) | (tt > 1 - 1e-4), axis=1)  # the fp32 lookup may read the neighbour cell
    rel = np.abs(got[:, 3] - ref) / ref
    assert np.all(rel[~near_edge] < 1e-4) and near_edge.mean() < 1e-2
    assert np.all(rel < 1e-6)       # the sampler returns the density of the cell it drew, at a cell edge too
    # round trip, bit for bit, wherever the fp32 direction reads back the cell it was drawn in
    back = sc.env_pdf(got[:, :3])
    assert np.array_equal(back[~near_edge], got[~near_edge, 3]) and (back != got[:, 3]).mean() < 1e-3
    d = rng.normal(size=(20000, 3))
    p = sc.env_pdf(d)
    x, y = t.coords(d)
    edge = (np.abs(x - np.round(x)) < 1e-4) | (np.abs(y - np.round(y)) < 1e-4)
    pr = t.pdf(d)
    assert np.all(np.abs(p - pr)[~edge] <= 1e-4 * pr[~edge])
    sc.close()


@pytest.mark.gpu
def test_black_map_renders_without_shadow_rays(native_built):
    spec = scenes.diffuse_single_sphere(32, 32)
    sc = spec.scene(api.Image(16, 8, np.zeros((8, 16, 3))))
    with pytest.raises(_ffi.RayrsError):
        sc.env_sample(np.zeros((1, 2)))
    assert np.all(sc.env_pdf(np.eye(3)) == 0)
    img = api.render_gpu(spec.camera(), sc, 4, 8, flags=api.RRS_FLAG_ENV_SAMPLING)
    assert np.all(img == 0) and sc.stats()["census_mismatch_pixels"] == 0
    sc.close()


SEEDS_ON = [101 + k for k in range(12)]
SEEDS_OFF = [201 + k for k in range(12)]


@pytest.mark.gpu
def test_unbiased_config1(native_built, hdri_small):
    spec = scenes.diffuse_single_sphere(128, 128)
    sc = spec.scene(hdri_small)
    cam = spec.camera()
    on = _renders(sc, cam, 64, 8, api.RRS_FLAG_ENV_SAMPLING, SEEDS_ON)
    assert sc.stats()["kernel_form"] == _ffi.RRS_FORM_WAVEFRONT
    off = _renders(sc, cam, 64, 8, 0, SEEDS_OFF)
    print("config 1: worst |z| %.2f (bound %.2f)" % assert_same_mean(on, off))
    sc.close()


@pytest.mark.gpu
@pytest.mark.parametrize("sun", [2000.0, 20.0])
def test_unbiased_sun_scene(sun, native_built):
    """Lambertian + rough Cook-Torrance under an unclipped sun 2000 x the sky, and the same at 20 x: there the
    flag-off noise is low enough that a bias of 1 % of a block shows."""
    spec = scenes.sun_spheres()
    sc = spec.scene(scenes.sun_hdri(sun=sun))
    cam = spec.camera()
    seeds_on, seeds_off = [401 + k for k in range(32)], [501 + k for k in range(32)]
    on = _renders(sc, cam, 256, spec.max_bounces, api.RRS_FLAG_ENV_SAMPLING, seeds_on)
    off = _renders(sc, cam, 256, spec.max_bounces, 0, seeds_off)
    print("sun scene (sun %g x sky): worst |z| %.2f (bound %.2f)" % ((sun,) + assert_same_mean(on, off)))
    sc.close()


@pytest.mark.gpu
def test_unbiased_white_furnace(native_built):
    spec = _furnace_spec()
    sc = spec.scene(api.Image(32, 16, np.ones((16, 32, 3))))
    cam = spec.camera()
    on = _renders(sc, cam, 64, spec.max_bounces, api.RRS_FLAG_ENV_SAMPLING, SEEDS_ON[:8])
    off = _renders(sc, cam, 64, spec.max_bounces, 0, SEEDS_OFF[:8])
    assert np.allclose(off, 1.0, rtol=1e-6)   # albedo 1 under a uniform 1: every path returns exactly 1
    assert abs(on.mean() - 1.0) < 1e-3
    assert_same_mean(on, off)
    sc.close()


@pytest.mark.gpu
def test_variance_is_lower_on_the_sun_scene(sun_scene):
    spec, sc = sun_scene
    cam = spec.camera()
    seeds = [301 + k for k in range(8)]
    on = _renders(sc, cam, 64, spec.max_bounces, api.RRS_FLAG_ENV_SAMPLING, seeds)
    off = _renders(sc, cam, 64, spec.max_bounces, 0, seeds)
    v_on, v_off = on.sum(axis=3).var(axis=0, ddof=1).mean(), off.sum(axis=3).var(axis=0, ddof=1).mean()
    print(f"sun scene, 64 spp: mean per-pixel variance {v_off:.4g} -> {v_on:.4g} ({v_off / v_on:.1f}x lower)")
    assert v_on * 20 < v_off   # measured 171 x on a B200 (seeds 301..308)


@pytest.mark.gpu
def test_bvh_form_and_flag_combinations(native_built, hdri_small):
    """The BVH form of the env kernel (a mesh scene) converges to the flag-off image too; the path-loop request is
    overridden and the split form is refused."""
    spec = scenes.copper_torus(24, 12, 64, 48)
    sc = spec.scene(hdri_small)
    cam = spec.camera()
    on = _renders(sc, cam, 64, 16, api.RRS_FLAG_ENV_SAMPLING, SEEDS_ON[:8])
    off = _renders(sc, cam, 64, 16, 0, SEEDS_OFF[:8])
    assert_same_mean(on, off)
    with pytest.raises(_ffi.RayrsError):
        api.render_gpu(cam, sc, 4, 8, flags=api.RRS_FLAG_ENV_SAMPLING | _ffi.RRS_FLAG_SPLIT_KERNELS)
    sc.close()
    small = scenes.diffuse_single_sphere(32, 32)
    sc = small.scene(hdri_small)
    api.render_gpu(small.camera(), sc, 4, 8, flags=api.RRS_FLAG_ENV_SAMPLING | _ffi.RRS_FLAG_FORCE_PATHLOOP)
    assert sc.stats()["kernel_form"] == _ffi.RRS_FORM_WAVEFRONT
    sc.close()


@pytest.mark.gpu
def test_multi_gpu_matches_one_gpu(native_built, hdri_small):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    spec = scenes.diffuse_single_sphere(64, 64)
    one = spec.scene(hdri_small)
    two = spec.scene(hdri_small, devices=[0, 1])
    cam = spec.camera()
    a = api.render_gpu(cam, one, 32, 8, flags=api.RRS_FLAG_ENV_SAMPLING).astype(np.float64)
    b = api.render_gpu(cam, two, 32, 8, flags=api.RRS_FLAG_ENV_SAMPLING).astype(np.float64)
    assert np.max(np.abs(a - b) / np.maximum(np.abs(a), 1e-3)) <= 1e-6
    one.close()
    two.close()
