"""Environment sampling (RRS_FLAG_ENV_SAMPLING) held to the f64 oracle's restatement of the same estimator.

The oracle (oracle.cpp: build_env_table, env_sample, nee_bsdf, radiance with env) draws the same Philox uniforms as
the device, so with RNG_MATCHED the two trace the same paths and shadow rays, and an ENV image must agree with the
oracle's ENV render far below the Monte-Carlo noise: a change to the estimator shows at rounding level.

CPU: the oracle's table equals the numpy restatement of test_env_sampling bit for bit, its sampler and density agree
with it, its ENV estimator converges to its plain render (f64, many samples), and in a closed box it changes nothing
but the ray count.
GPU: sample-matched ENV images on opaque scenes, statistical agreement on transmissive ones (the SPH64 kernels),
invariances that hold up to fp32 summation order, and the refusal of maps with non-finite texels.
"""
import numpy as np
import pytest

import oracle
from conftest import relrmse
from rayrs_b200 import _ffi, api, scenes
from test_env_sampling import EnvTable, _furnace_spec, assert_same_mean, background_np, hot_texel_map

ENV = api.RRS_FLAG_ENV_SAMPLING


def _oracle(spec, pixels):
    return oracle.OracleScene(spec.tables(), pixels, heuristic=(spec.heuristic.kind, spec.heuristic.splits), build_mode=1)


def _map(name):
    rng = np.random.default_rng(sum(map(ord, name)))
    if name == "synthetic":
        return scenes.synthetic_hdri(128, 64).pixels
    if name == "sun":
        return scenes.sun_hdri().pixels
    if name == "sun_1e12":                      # sky 1e-6, sun 1e6: the one-step minimum decides the sky's cells
        return scenes.sun_hdri(sky=1e-6, sun=1e6).pixels
    if name == "hot_texel":
        return hot_texel_map()
    if name in ("2x2", "3x2", "37x19"):
        w, h = map(int, name.split("x"))
        return rng.uniform(0.1, 4.0, size=(h, w, 3))
    if name == "negative":                      # |texel| weighs the table; background() may be negative
        return rng.uniform(0.1, 2.0, size=(16, 24, 3)) * rng.choice([-1.0, 1.0], size=(16, 24, 3))
    px = np.zeros((16, 24, 3))
    if name == "row0":
        px[0] = (3.0, 2.0, 1.0)
    elif name == "row_last":
        px[-1] = (1.0, 2.0, 3.0)
    elif name == "col0":
        px[:, 0] = (2.0, 0.0, 0.0)
    elif name == "col_last":
        px[:, -1] = (0.0, 0.0, 5.0)
    elif name == "pole_sun":                    # the sun in the pole row (cells of the smallest solid angle)
        px[:] = 1.0
        px[0, 7:10] = (2000.0, 1900.0, 1700.0)
    else:
        raise KeyError(name)
    return px


MAPS = ["synthetic", "sun", "hot_texel", "2x2", "3x2", "37x19", "row0", "row_last", "col0", "col_last", "negative",
        "sun_1e12", "pole_sun"]
_TABLE_SCENE = scenes.diffuse_single_sphere(8, 8)


# ---------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", MAPS)
def test_oracle_table_equals_restatement(name):
    px = _map(name)
    osc = _oracle(_TABLE_SCENE, px)
    got = osc.env_table()
    t = EnvTable(px)
    assert np.array_equal(got["marg"], t.marg)
    assert np.array_equal(got["cond"], t.cond)
    assert np.array_equal(got["row"][:, 0], t.cos0) and np.array_equal(got["row"][:, 1], t.dcos)
    osc.close()


def test_oracle_table_black_and_non_finite_maps():
    osc = _oracle(_TABLE_SCENE, np.zeros((8, 16, 3)))
    assert osc.env_table() is None
    assert np.all(osc.env_pdf(np.eye(3)) == 0)
    with pytest.raises(ValueError):
        osc.env_sample(np.zeros((1, 2)))
    osc.close()
    for ch, v in ((0, np.nan), (1, np.nan), (2, np.nan), (1, np.inf), (2, -np.inf)):
        px = np.ones((8, 16, 3))
        px[3, 5, ch] = v
        osc = _oracle(_TABLE_SCENE, px)
        for call in (osc.env_table, lambda: osc.env_pdf(np.eye(3)), lambda: osc.env_sample(np.zeros((1, 2)))):
            with pytest.raises(ValueError):
                call()
        osc.close()


@pytest.mark.parametrize("name", MAPS)
def test_oracle_sampler_equals_restatement(name):
    px = _map(name)
    osc = _oracle(_TABLE_SCENE, px)
    t = EnvTable(px)
    rng = np.random.default_rng(11)
    G = float(1 << 24)
    edge_u = np.array([0.0, 1.0 - 2.0 ** -53, 0.5, 1.0 / G, 1.0 - 1.0 / G, 0.25 - 2.0 ** -40])
    u = np.concatenate([rng.random((20000, 2)), np.stack(np.meshgrid(edge_u, edge_u), -1).reshape(-1, 2),
                        t.marg[rng.integers(0, t.ch, 64)].astype(np.float64)[:, None] * np.ones((1, 2))])
    got = osc.env_sample(u)
    dirs, i, j, tt = t.sample(u)
    assert np.array_equal(got[:, 4].astype(np.int64), i) and np.array_equal(got[:, 5].astype(np.int64), j)
    assert np.max(np.abs(got[:, :3] - dirs)) < 1e-12
    assert np.array_equal(got[:, 3], t.cell_pdf[i, j])           # the density of the drawn cell
    # env_pdf reads the cell background() reads: the same cell except within 1e-9 of a cell edge, and within the fp32
    # rounding of the table's row edges (cos theta is stored in fp32: 1e-6 of the cell's extent)
    x, y = t.coords(got[:, :3])
    edge = (np.abs(x - np.round(x)) < 1e-9) | (np.abs(y - np.round(y)) < 1e-9) | np.any((tt < 1e-6) | (tt > 1 - 1e-6), axis=1)
    p = osc.env_pdf(got[:, :3])
    assert np.array_equal(p[~edge], got[~edge, 3])
    assert edge.mean() < 0.01
    # and the density lookup of arbitrary directions is the restatement's
    d = rng.normal(size=(20000, 3))
    x, y = t.coords(d)
    edge = (np.abs(x - np.round(x)) < 1e-9) | (np.abs(y - np.round(y)) < 1e-9)
    assert np.array_equal(osc.env_pdf(d)[~edge], t.pdf(d)[~edge])
    # the density is positive wherever the background is not zero
    lit = np.abs(background_np(px, d)).max(axis=1) > 0
    assert np.all(osc.env_pdf(d)[lit] > 0)
    osc.close()


def _oracle_renders(osc, cam, spp, mb, env, seeds):
    W, H = cam.x_pixels(), cam.y_pixels()
    out = []
    for s in seeds:
        img, st = osc.render(cam.derived17(), W, H, spp, max_bounces=mb, seed=s, rng_mode=oracle.RNG_WIDE, env=env)
        assert st["nan_pixels"] == 0
        assert not env or st["shadow_rays"] > 0
        out.append(img)
    return np.stack(out)


UNBIASED = {
    # name: (spec builder, map, spp, max_bounces)
    "sun_2000": (lambda: scenes.sun_spheres(24, 16), lambda: scenes.sun_hdri().pixels, 256, 16),
    "sun_20": (lambda: scenes.sun_spheres(24, 16), lambda: scenes.sun_hdri(sun=20.0).pixels, 256, 16),
    "metallic_alpha_0.01": (lambda: scenes.cook_torrance_spheres_metallic(64, 16), lambda: scenes.synthetic_hdri(128, 64).pixels, 256, 16),
}


@pytest.mark.parametrize("name", sorted(UNBIASED))
def test_oracle_env_estimator_is_unbiased(name):
    """The estimator's design, in f64 and without a GPU: the ENV render converges to the plain render (per 8 x 8 block,
    bound from the standard errors measured over independent seeds)."""
    builder, hdri, spp, mb = UNBIASED[name]
    spec = builder()
    osc = _oracle(spec, hdri())
    cam = spec.camera()
    on = _oracle_renders(osc, cam, spp, mb, True, range(1, 17))
    off = _oracle_renders(osc, cam, spp, mb, False, range(101, 117))
    assert_same_mean(on, off)
    osc.close()


def test_oracle_env_white_furnace():
    spec = _furnace_spec(16, 16)
    osc = _oracle(spec, np.ones((16, 32, 3)))
    cam = spec.camera()
    off = _oracle_renders(osc, cam, 16, spec.max_bounces, False, [1])
    assert np.allclose(off, 1.0, rtol=1e-12)
    on = _oracle_renders(osc, cam, 64, spec.max_bounces, True, range(1, 5))
    se = on.std(ddof=1) / np.sqrt(on.size)
    assert abs(on.mean() - 1.0) < 4.0 * se + 1e-12, (on.mean(), se)
    osc.close()


def closed_box_spec(W=32, H=24):
    """The camera, an emitter and three materials inside a closed box: the environment is invisible.  The walls are six
    planes facing inwards that overlap at the edges.  (Object.box_geom repeats the reference's planes: its Y and YRev
    faces both lie at the lower y and its ZRev face looks outwards, so a scattered ray can leave it.)"""
    w, h = scenes.film(W, H)
    lo, hi, e = (-4.0, -1.0, -4.0), (4.0, 5.0, 6.0), 1.0
    wall = api.Material.lambertian_diffuse((0.7, 0.7, 0.7))
    A = api.Axis
    objects = [
        api.Object.plane(A.X, lo[1] - e, hi[1] + e, lo[2] - e, hi[2] + e, lo[0], wall),
        api.Object.plane(A.XRev, lo[1] - e, hi[1] + e, lo[2] - e, hi[2] + e, hi[0], wall),
        api.Object.plane(A.Y, lo[0] - e, hi[0] + e, lo[2] - e, hi[2] + e, lo[1], wall),
        api.Object.plane(A.YRev, lo[0] - e, hi[0] + e, lo[2] - e, hi[2] + e, hi[1], wall),
        api.Object.plane(A.Z, lo[0] - e, hi[0] + e, lo[1] - e, hi[1] + e, lo[2], wall),
        api.Object.plane(A.ZRev, lo[0] - e, hi[0] + e, lo[1] - e, hi[1] + e, hi[2], wall),
        api.Object.sphere(0.7, (-1.5, 0.7, 0.0), wall, api.Emission.new(5.0, (1.0, 0.8, 0.6))),
        api.Object.sphere(0.8, (1.2, 0.8, 0.2), api.Material.cook_torrance((1, 1, 1), 0.1, api.Fresnel.schlick_metallic((0.9, 0.6, 0.3)))),
        api.Object.sphere(0.5, (0.0, 0.5, 1.5), api.Material.plastic((0.2, 0.5, 0.8), (1, 1, 1), 0.1, 1.45)),
    ]
    cam = dict(origin=(0.0, 2.5, 5.0), up=(0.0, 1.0, 0.0), lookat=(0.0, 0.8, 0.0), fov=60.0, width=w, height=h, ppi=scenes.PPI)
    return scenes.SceneSpec("closed_box", cam, objects, api.BvhHeuristic.Sah(1000), max_bounces=8)


def test_oracle_closed_box_hides_the_environment():
    spec = closed_box_spec()
    cam = spec.camera()
    osc = _oracle(spec, scenes.sun_hdri().pixels)
    W, H = cam.x_pixels(), cam.y_pixels()
    off, so = osc.render(cam.derived17(), W, H, 16, max_bounces=spec.max_bounces)
    on, sn = osc.render(cam.derived17(), W, H, 16, max_bounces=spec.max_bounces, env=True)
    assert off.max() > 0
    assert np.array_equal(on, off)
    assert sn["shadow_rays"] > 0 and sn["rays"] - so["rays"] == sn["shadow_rays"]
    osc.close()


# ---------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------
def _stats_ok(st):
    assert st["census_mismatch_pixels"] == 0 and st["nan_pixels"] == 0 and st["negative_pixels"] == 0, st


def _sky_2x2():
    return api.Image(2, 2, np.array([[[0.9, 1.0, 1.2], [3.0, 2.5, 2.0]], [[0.3, 0.25, 0.2], [0.6, 0.5, 0.4]]]))


def _pole_sun():
    return api.Image(24, 16, _map("pole_sun"))


MATCHED = {
    # name: (spec builder, map builder (None: the shared hdri_small), spp, max_bounces)
    "config1": (lambda: scenes.diffuse_single_sphere(96, 96), None, 32, 8),
    "sun_spheres_2000": (lambda: scenes.sun_spheres(64, 48), lambda: scenes.sun_hdri(), 64, 16),
    "spheres_metallic": (lambda: scenes.cook_torrance_spheres_metallic(240, 96), None, 32, 50),
    "spheres_plastic": (lambda: scenes.cook_torrance_spheres_plastic(240, 96), None, 32, 50),
    "emissive_room": (lambda: scenes.emissive_room(240, 160), None, 32, 50),
    "copper_torus": (lambda: scenes.copper_torus(24, 12, 96, 64), None, 32, 16),
    "sun_spheres_map_2x2": (lambda: scenes.sun_spheres(64, 48), _sky_2x2, 32, 16),
    "sun_spheres_pole_sun": (lambda: scenes.sun_spheres(64, 48), _pole_sun, 32, 16),
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(MATCHED))
def test_env_sample_matched_image(name, hdri_small):
    """The protocol of test_gpu_render.test_sample_matched_image, with the flag on both sides: the same paths and the
    same shadow rays, so the residual is fp32 rounding plus the rare decision that flips."""
    builder, hdri, spp, mb = MATCHED[name]
    spec = builder()
    img_map = hdri() if hdri else hdri_small
    sc, osc, cam = spec.scene(img_map), _oracle(spec, img_map.pixels), spec.camera()
    W, H = cam.x_pixels(), cam.y_pixels()
    img = api.render_gpu(cam, sc, spp, mb, flags=ENV).astype(np.float64)
    st = sc.stats()
    ref, ost = osc.render(cam.derived17(), W, H, spp, max_bounces=mb, env=True)
    noise, _ = osc.render(cam.derived17(), W, H, spp, max_bounces=mb, seed=999, env=True)
    e, e0 = relrmse(img, ref), relrmse(noise, ref)
    rel = np.abs(img - ref).max(axis=2) / (np.abs(ref).max(axis=2) + 0.1)
    print(f"[{name}] relRMSE matched {e:.3e} vs noise floor {e0:.3e} (ratio {e / e0:.2e}); pixels off by >1e-3: "
          f"{(rel > 1e-3).sum()} of {rel.size}; rays gpu {st['rays']} oracle {ost['rays']} "
          f"(rel {(st['rays'] - ost['rays']) / ost['rays']:+.2e}); shadow rays {ost['shadow_rays']}")
    assert ost["shadow_rays"] > 0
    assert e < 0.02 * e0, (e, e0)
    assert (rel > 1e-3).mean() < 0.01
    assert abs(st["rays"] - ost["rays"]) <= 2e-4 * ost["rays"]
    assert st["paths"] == W * H * spp
    _stats_ok(st)
    assert ost["nan_pixels"] == 0
    sc.close()
    osc.close()


TRANSMISSIVE = {
    "material_test": (lambda: scenes.material_test(280, 56), 64),
    "glass_single_sphere": (lambda: scenes.glass_single_sphere(160, 96), 64),
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(TRANSMISSIVE))
def test_env_transmissive_statistical(name, hdri_small):
    """Transmissive spheres run the SPH64 instantiations of the ENV kernel; their f64 re-entry coin flip cannot be
    matched ray by ray, so the protocol of test_gpu_render.test_statistical_image applies, against the oracle's ENV
    render: within the oracle-vs-oracle noise, per-object means within their standard errors, and the distance at 4x
    the samples shrinking like noise."""
    builder, spp = TRANSMISSIVE[name]
    spec = builder()
    sc, osc, cam = spec.scene(hdri_small), _oracle(spec, hdri_small.pixels), spec.camera()
    W, H = cam.x_pixels(), cam.y_pixels()
    c17 = cam.derived17()
    A, sa = osc.render(c17, W, H, spp, seed=101, rng_mode=oracle.RNG_WIDE, env=True)
    B, _ = osc.render(c17, W, H, spp, seed=202, rng_mode=oracle.RNG_WIDE, env=True)
    G = api.render_gpu(cam, sc, spp, 50, seed=303, flags=ENV).astype(np.float64)
    _stats_ok(sc.stats())
    assert sa["shadow_rays"] > 0
    e0, eg = relrmse(A, B), relrmse(G, A)
    assert eg <= 1.25 * e0, (eg, e0)
    rows, cols = np.mgrid[0:H, 0:W]
    pr = oracle.primary_rays(c17, W, H, rows.ravel(), cols.ravel(), np.zeros(W * H, dtype=np.uint32))
    ids = osc.intersect(pr)[0].reshape(H, W)
    worst = 0.0
    for k in range(-1, min(int(ids.max()) + 1, 8)):
        mask = ids == k
        if mask.sum() < 200:
            continue
        se = np.sqrt((((A[mask] - B[mask]) ** 2) / 2.0).sum(axis=0)) / mask.sum()
        z = np.abs(G[mask].mean(axis=0) - A[mask].mean(axis=0)) / (np.sqrt(2.0) * se + 1e-12)
        worst = max(worst, float(z.max()))
        assert (z < 4.5).all(), (name, k, z)
    A4, _ = osc.render(c17, W, H, 4 * spp, seed=404, rng_mode=oracle.RNG_WIDE, env=True)
    G4 = api.render_gpu(cam, sc, 4 * spp, 50, seed=505, flags=ENV).astype(np.float64)
    eg4 = relrmse(G4, A4)
    print(f"[{name}] ENV relRMSE gpu-vs-oracle {eg:.4f} (noise floor {e0:.4f}); at 4x spp {eg4:.4f} "
          f"(ratio {eg4 / eg:.3f}); worst region z {worst:.2f}")
    assert eg4 < 0.65 * eg, (eg4, eg)
    sc.close()
    osc.close()


@pytest.mark.gpu
def test_env_invariances(native_built):
    """A ragged 37 x 19 image of a three-primitive scene under an unclipped sun: the ENV image does not depend on the
    queue size, on the kernel form (brute force / BVH), or on splitting the samples into ranges (shadow rays do not
    count as path ends), up to fp32 summation order; it matches the oracle at every depth."""
    import torch
    spec = scenes.sun_spheres(37, 19)
    hdri = scenes.sun_hdri(sun=20.0)
    sc, osc, cam = spec.scene(hdri), _oracle(spec, hdri.pixels), spec.camera()
    c17 = cam.derived17()
    W, H, spp, mb = 37, 19, 40, spec.max_bounces
    assert (cam.x_pixels(), cam.y_pixels()) == (W, H)
    base = api.render_gpu(cam, sc, spp, mb, flags=ENV).astype(np.float64)
    st0 = sc.stats()
    _stats_ok(st0)
    ref, ost = osc.render(c17, W, H, spp, max_bounces=mb, env=True)
    noise, _ = osc.render(c17, W, H, spp, max_bounces=mb, seed=999, env=True)
    assert relrmse(base, ref) < 0.02 * relrmse(noise, ref)
    assert abs(st0["rays"] - ost["rays"]) <= 2e-4 * ost["rays"]
    for q in (1024, 4096, 1 << 16):
        img = api.render_gpu(cam, sc, spp, mb, queue_capacity=q, flags=ENV).astype(np.float64)
        st = sc.stats()
        _stats_ok(st)
        assert st["rays"] == st0["rays"], q
        assert np.allclose(img, base, rtol=2e-5, atol=1e-6), q
    # the same scene in the BVH form of the kernel
    bvh = spec.scene(hdri, scene_flags=_ffi.RRS_SCENE_NO_BRUTE)
    img = api.render_gpu(cam, bvh, spp, mb, flags=ENV).astype(np.float64)
    assert bvh.stats()["rays"] == st0["rays"]
    assert np.allclose(img, base, rtol=2e-5, atol=1e-6)
    bvh.close()
    # four sample ranges accumulated into one buffer: every pixel ends exactly spp paths
    acc = torch.zeros((H, W, 4), dtype=torch.float32, device="cuda:0")
    stream = torch.cuda.current_stream().cuda_stream
    rays = 0
    for g in range(4):
        api.render_accumulate(cam, sc, spp // 4, mb, acc.data_ptr(), stream, sample_offset=g * (spp // 4), spp_total=spp,
                              flags=ENV)
        rays += sc.stats()["rays"]
    torch.cuda.synchronize()
    a = acc.cpu().numpy().astype(np.float64)
    assert np.array_equal(a[..., 3], np.full((H, W), float(spp)))
    assert rays == st0["rays"]
    assert np.allclose(a[..., :3] / spp, base, rtol=2e-5, atol=1e-6)
    # max_bounces = 1: no vertex may emit a shadow ray (the image is the camera rays' escapes)
    one_on = api.render_gpu(cam, sc, 8, 1, flags=ENV).astype(np.float64)
    r_on = sc.stats()["rays"]
    one_off = api.render_gpu(cam, sc, 8, 1).astype(np.float64)
    assert r_on == sc.stats()["rays"] == W * H * 8
    assert np.allclose(one_on, one_off, rtol=2e-5, atol=1e-6)
    # depth 2 and 3 against the oracle, ray for ray
    for d in (2, 3):
        img = api.render_gpu(cam, sc, 16, d, flags=ENV).astype(np.float64)
        st = sc.stats()
        r, o = osc.render(c17, W, H, 16, max_bounces=d, env=True)
        print(f"[invariances] depth {d}: rays gpu {st['rays']} oracle {o['rays']} (shadow {o['shadow_rays']}); "
              f"relRMSE {relrmse(img, r):.2e}")
        assert o["shadow_rays"] > 0 and st["rays"] == o["rays"], d
        assert relrmse(img, r) < 5e-3
    sc.close()
    osc.close()


@pytest.mark.gpu
def test_env_closed_box(native_built):
    """Inside a closed box every shadow ray is blocked: flag on and off render the same image, and the device traces
    as many more rays with the flag as the oracle's shadow-ray count."""
    spec = closed_box_spec()
    hdri = scenes.sun_hdri()
    sc, osc, cam = spec.scene(hdri), _oracle(spec, hdri.pixels), spec.camera()
    W, H = cam.x_pixels(), cam.y_pixels()
    off = api.render_gpu(cam, sc, 32, spec.max_bounces).astype(np.float64)
    r_off = sc.stats()["rays"]
    on = api.render_gpu(cam, sc, 32, spec.max_bounces, flags=ENV).astype(np.float64)
    st = sc.stats()
    _stats_ok(st)
    _, o = osc.render(cam.derived17(), W, H, 32, max_bounces=spec.max_bounces, env=True)
    print(f"[closed box] rays off {r_off}, on {st['rays']}; oracle shadow rays {o['shadow_rays']}")
    assert off.max() > 0
    assert np.allclose(on, off, rtol=2e-5, atol=1e-6)
    assert abs((st["rays"] - r_off) - o["shadow_rays"]) <= 2e-4 * o["rays"]
    sc.close()
    osc.close()


@pytest.mark.gpu
@pytest.mark.parametrize("channel,value", [(0, np.nan), (1, np.nan), (2, np.nan), (1, np.inf), (2, -np.inf)])
def test_env_refuses_non_finite_maps(channel, value, native_built):
    px = np.ones((16, 32, 3))
    px[5, 9, channel] = value
    spec = scenes.diffuse_single_sphere(32, 32)
    sc = spec.scene(api.Image(32, 16, px))
    api.render_gpu(spec.camera(), sc, 4, 8)                     # the plain render takes the map as it is
    with pytest.raises(_ffi.RayrsError) as e:
        api.render_gpu(spec.camera(), sc, 4, 8, flags=ENV)
    assert e.value.status == _ffi.RRS_ERR_INVALID
    with pytest.raises(_ffi.RayrsError):
        sc.env_sample(np.zeros((1, 2)))
    with pytest.raises(_ffi.RayrsError):
        sc.env_pdf(np.eye(3))
    sc.close()
