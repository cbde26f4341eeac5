"""T3 — texture::value(u, v, p) on the device vs the oracle: checker / image are integer
decisions (exact away from cell / texel borders), Perlin marble within fp32 tolerance."""
import numpy as np
import pytest

import scene_util as su

pytestmark = pytest.mark.gpu
NOISE_ATOL = 5e-4  # fp32 7-octave turbulence inside sin(); stated tolerance for T3


def _points(rng, n, span):
    uvp = np.empty((n, 5))
    uvp[:, :2] = rng.uniform(-0.2, 1.2, (n, 2))
    uvp[:, 2:] = rng.uniform(-span, span, (n, 3))
    return uvp


def test_solid_checker_nested_checker(rtb, orc, gpu_ctx):
    rng = np.random.default_rng(1)
    s = su.SceneDesc()
    a, b, c = s.solid(0.2, 0.3, 0.1), s.solid(0.9, 0.9, 0.9), s.solid(0.1, 0.2, 0.9)
    chk = s.checker(0.32, a, b)
    nested = s.checker(2.0, chk, c)
    desc = s.finish(s.sphere((0, 0, 0), 1, s.lambertian(nested)))
    gpu_ctx.upload_scene(desc)
    uvp = _points(rng, 200_000, 20.0)
    for tex in (a, chk, nested):
        got = gpu_ctx.eval_texture(tex, uvp)
        want = orc.texture_value(desc, tex, uvp)
        same = np.all(np.abs(got - want) < 1e-6, axis=1)
        assert same.mean() >= 0.9999  # only points within fp32 eps of a cell border may flip
    # negative coordinates: C++ remainder semantics (-1 % 2 == -1 -> odd), SURVEY A.17
    pts = np.array([[0, 0, -0.1, 0.1, 0.1], [0, 0, -0.1, -0.1, 0.1], [0, 0, -0.5, -0.5, -0.5]])
    assert np.allclose(gpu_ctx.eval_texture(chk, pts), orc.texture_value(desc, chk, pts), atol=1e-6)


def test_image_texture_nearest_texel_and_failed_load(rtb, orc, gpu_ctx):
    rng = np.random.default_rng(2)
    img = rng.integers(0, 256, (37, 53, 3), dtype=np.uint8)
    s = su.SceneDesc()
    t_img = s.image(img)
    t_bad = s.image(None)
    desc = s.finish(s.sphere((0, 0, 0), 1, s.lambertian(t_img)))
    gpu_ctx.upload_scene(desc)
    uvp = _points(rng, 200_000, 1.0)  # u, v outside [0,1] are clamped (texture.hpp:106-108)
    got = gpu_ctx.eval_texture(t_img, uvp)
    want = orc.texture_value(desc, t_img, uvp)
    same = np.all(np.abs(got - want) < 1e-6, axis=1)
    assert same.mean() >= 0.999
    # texel centres are unambiguous: exact
    jj, ii = np.meshgrid(np.arange(37), np.arange(53), indexing="ij")
    c = np.zeros((37 * 53, 5))
    c[:, 0] = (ii.ravel() + 0.5) / 53
    c[:, 1] = 1.0 - (jj.ravel() + 0.5) / 37
    assert np.allclose(gpu_ctx.eval_texture(t_img, c), orc.texture_value(desc, t_img, c), atol=1e-7)
    assert np.allclose(gpu_ctx.eval_texture(t_img, c).reshape(37, 53, 3), img / np.float32(255.0), atol=1e-6)
    # u == 1.0 / v == 0.0 hit the "high - 1" clamp (rtw_stb_image.hpp:123-134)
    edge = np.array([[1.0, 0.0, 0, 0, 0], [0.0, 1.0, 0, 0, 0], [1.0, 1.0, 0, 0, 0]])
    assert np.allclose(gpu_ctx.eval_texture(t_img, edge), orc.texture_value(desc, t_img, edge), atol=1e-7)
    # failed load -> cyan (texture.hpp:100-103)
    assert np.allclose(gpu_ctx.eval_texture(t_bad, uvp[:10]), [[0, 1, 1]] * 10)


def test_perlin_marble(rtb, orc, gpu_ctx):
    rng = np.random.default_rng(3)
    s = su.SceneDesc()
    t4, t02 = s.noise(4.0, rng), s.noise(0.2, rng)
    desc = s.finish(s.sphere((0, 0, 0), 1, s.lambertian(t4)))
    gpu_ctx.upload_scene(desc)
    for tex, span in ((t4, 6.0), (t02, 300.0)):
        uvp = _points(rng, 100_000, span)
        got = gpu_ctx.eval_texture(tex, uvp)
        want = orc.texture_value(desc, tex, uvp)
        err = np.abs(got - want).max(axis=1)
        assert np.quantile(err, 0.999) <= NOISE_ATOL, np.quantile(err, 0.999)
        assert err.mean() <= 5e-5


def test_earth_texture_through_named_scene(rtb, orc, gpu_ctx, earthmap):
    """The earth scene's earthmap.jpg (the reference's or the stand-in, conftest.py) through the host JPEG decoder + rtw_image conventions."""
    sc = rtb.Scene("earth", rand_seed=1)
    d = sc.desc.contents
    assert d.n_images == 1 and d.images[0].width == earthmap["width"] and d.images[0].height == earthmap["height"]
    gpu_ctx.upload_scene(sc.desc)
    rng = np.random.default_rng(4)
    uvp = _points(rng, 100_000, 1.0)
    tex = [i for i in range(d.n_textures) if d.textures[i].kind == rtb.RT_T_IMAGE][0]
    got = gpu_ctx.eval_texture(tex, uvp)
    want = orc.texture_value(sc.desc, tex, uvp)
    assert np.all(np.abs(got - want) < 1e-6, axis=1).mean() >= 0.999


def test_textured_phase_function_of_a_medium(rtb, orc, gpu_ctx):
    """constant_medium with a TEXTURED isotropic phase function (the book only ever uses a solid colour, and its medium
    hit leaves rec.u / rec.v unset): this repo defines u = v = 0 for a medium hit — device surface_at, oracle.cpp and
    oracle/ref_ext.hpp alike — so an image texture reads its (u, v) = (0, 0) texel and a checker follows the scatter
    point.  The converged GPU image must match the oracle's for both."""
    rng = np.random.default_rng(5)
    img = np.zeros((4, 4, 3), np.uint8)
    img[:] = (40, 200, 90)
    img[3, 0] = (250, 60, 20)  # the texel at (u, v) = (0, 0): v is flipped (texture.hpp:109), row 3
    for kind in ("image", "checker"):
        s = su.SceneDesc()
        tex = s.image(img) if kind == "image" else s.checker(1.3, s.solid(0.9, 0.2, 0.1), s.solid(0.1, 0.3, 0.9))
        fog = s.medium(s.sphere((0, 0, 0), 2.0, s.dielectric(1.5)), 1.5, s.isotropic(tex))
        floor = s.quad((-6, -2.2, -6), (12, 0, 0), (0, 0, 12), s.lambertian(s.solid(0.5, 0.5, 0.5)))
        desc = s.finish(s.list([fog, floor]))
        cam = su.camera(width=64, spp=2048, depth=12, lookfrom=(0, 1, 9), vfov=35.0)
        gpu_ctx.upload_scene(desc)
        gpu_ctx.render(cam, seed=3)
        got = gpu_ctx.download_radiance(cam.samples_per_pixel).astype(np.float64)
        mean, var, _ = orc.render_linear(desc, cam, spp=256, seed=9)
        var_tot = var * (1.0 + 256 / 2048)
        for c in range(3):
            z = (got[..., c].sum() - mean[..., c].sum()) / np.sqrt(var_tot[..., c].sum() + 1e-30)
            assert abs(z) < 5.0, (kind, c, z)
        centre = got[24:40, 24:40].mean(axis=(0, 1))  # the fog ball: its colour is the texture's
        if kind == "image":
            assert centre[0] > 1.5 * centre[1], centre  # the reddish (0, 0) texel, not the green rest of the image
