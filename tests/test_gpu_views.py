"""rt_render_views / Context.render_views / rtb200::render_views: many camera views of one scene in one launch.

View v of a batch must have exactly the bits of rt_render(cams[v]) with the same seed and sample range — the
accumulator is an integer sum and the Philox counter is (in-view pixel, sample, bounce, stream), so no tolerance is
involved.  The single renders are the oracle."""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def orbit(rtb, sc, n, width, spp, depths=None):
    """n views on a circle about the scene camera's lookat (vertical axis), each with its own vfov, defocus,
    max_depth and background."""
    base = sc.cam.contents
    at = np.array(base.lookat[:])
    r = np.array(base.lookfrom[:]) - at
    depths = depths or [base.max_depth, 3, 1, 7, 12]
    bgs = [tuple(base.background[:]), (0.7, 0.8, 1.0), (0.1, 0.0, 0.05), (0.0, 0.0, 0.0), (1.0, 1.0, 1.0)]
    cams = []
    for v in range(n):
        a = 2.0 * math.pi * v / n
        c, s = math.cos(a), math.sin(a)
        frm = at + np.array([c * r[0] + s * r[2], r[1], -s * r[0] + c * r[2]])
        cams.append(sc.camera_copy(image_width=width, samples_per_pixel=spp, lookfrom=tuple(frm), vfov=base.vfov * (0.8 + 0.15 * v),
                                   defocus_angle=[0.0, 0.6, base.defocus_angle, 2.0][v % 4], max_depth=depths[v % len(depths)],
                                   background=bgs[v % len(bgs)]))
    return cams


def singles(ctx, cams, seed, **kw):
    """The oracle: every view through rt_render.  Returns (V, H, W, 3) sums, rays, samples."""
    acc, rays, samples = [], 0, 0
    for cam in cams:
        ctx.render(cam, seed=seed, **kw)
        acc.append(ctx.download_accum())
        st = ctx.stats()
        rays, samples = rays + st.rays, samples + st.samples
    return np.stack(acc), rays, samples


def batch(ctx, cams, seed, **kw):
    ctx.render_views(cams, seed=seed, **kw)
    st = ctx.stats()
    return ctx.download_accum(), st.rays, st.samples


def assert_same(got, want):
    acc, rays, samples = got
    assert acc.shape == want[0].shape
    for v in range(acc.shape[0]):
        assert np.array_equal(acc[v], want[0][v]), f"view {v}: {(acc[v] != want[0][v]).sum()} values differ"
    assert (rays, samples) == (want[1], want[2])


# bouncing_spheres: moving spheres, shared-memory stack; book1_final: defocus; book2_final: staged, local stack, fog;
# perlin_sphere: cooperative turbulence; cornell_smoke: box media; earth: image texture
@pytest.mark.parametrize("name,n", [("bouncing_spheres", 5), ("book1_final", 4), ("book2_final", 4), ("perlin_sphere", 3),
                                    ("cornell_smoke", 4), ("earth", 5)])
def test_views_equal_their_single_renders(rtb, gpu_ctx, name, n):
    sc = rtb.Scene(name, rand_seed=1)
    cams = orbit(rtb, sc, n, 64, 8)
    gpu_ctx.upload_scene(sc.desc)
    want = singles(gpu_ctx, cams, seed=11)
    got = batch(gpu_ctx, cams, seed=11)
    assert_same(got, want)
    assert got[0].any()


# every other launch plan: BVH top only in shared memory (not staged), local-memory stacks, each with and without the
# cooperative turbulence; the knobs are read when a context is created
@pytest.mark.parametrize("name,knob", [("bouncing_spheres", "RT_B200_NO_STAGING"), ("perlin_sphere", "RT_B200_NO_STAGING"),
                                       ("bouncing_spheres", "RT_B200_NO_SMEM_STACK"), ("perlin_sphere", "RT_B200_NO_SMEM_STACK")])
def test_views_equal_their_single_renders_under_every_plan(rtb, monkeypatch, name, knob):
    monkeypatch.setenv(knob, "1")
    ctx = rtb.Context(0)
    try:
        sc = rtb.Scene(name, rand_seed=1)
        cams = orbit(rtb, sc, 4, 48, 6)
        ctx.upload_scene(sc.desc)
        assert_same(batch(ctx, cams, seed=5), singles(ctx, cams, seed=5))
    finally:
        ctx.close()


@pytest.mark.parametrize("width,aspect,n,spp", [(37, 1.3, 3, 7), (13, 0.77, 4, 5), (50, 1.0, 1, 9), (24, 1.5, 256, 4)])
def test_shapes_ragged_single_and_large_batches(rtb, gpu_ctx, width, aspect, n, spp):
    """Sizes that are not multiples of the 8 x 4 tile, V = 1, and 256 views of 24 x 16."""
    sc = rtb.Scene("cornell_box", rand_seed=1)
    cams = orbit(rtb, sc, n, width, spp, depths=[6, 2, 9])
    for c in cams:
        c.aspect_ratio = aspect
    gpu_ctx.upload_scene(sc.desc)
    got = batch(gpu_ctx, cams, seed=2)
    assert got[0].shape == (n, rtb.image_height(cams[0]), width, 3)
    assert_same(got, singles(gpu_ctx, cams, seed=2))


def test_views_without_depth_trace_nothing(rtb, gpu_ctx):
    """max_depth <= 0: no path is traced for that view (as rt_render does nothing), its samples still count."""
    sc = rtb.Scene("bouncing_spheres", rand_seed=1)
    cams = orbit(rtb, sc, 6, 40, 6, depths=[5, 0, 3, -2, 0, 8])
    gpu_ctx.upload_scene(sc.desc)
    got = batch(gpu_ctx, cams, seed=4)
    assert_same(got, singles(gpu_ctx, cams, seed=4))
    for v in (1, 3, 4):
        assert not got[0][v].any()
    assert got[2] == 6 * 40 * rtb.image_height(cams[0]) * 6


def test_sample_ranges_and_forced_launch_splits_equal_one_call(rtb, gpu_ctx, monkeypatch):
    sc = rtb.Scene("book1_final", rand_seed=1)
    cams = orbit(rtb, sc, 4, 40, 24)
    gpu_ctx.upload_scene(sc.desc)
    whole = batch(gpu_ctx, cams, seed=8)
    # a batch rendered as sample ranges [0, 5) [5, 17) [17, 24), the later ones with clear = 0
    gpu_ctx.render_views(cams, seed=8, sample_begin=0, sample_count=5)
    gpu_ctx.render_views(cams, seed=8, sample_begin=5, sample_count=12, clear=False)
    gpu_ctx.render_views(cams, seed=8, sample_begin=17, sample_count=7, clear=False)
    st = gpu_ctx.stats()
    assert_same((gpu_ctx.download_accum(), st.rays, st.samples), whole)
    # the same range of a single render
    part = singles(gpu_ctx, cams, seed=8, sample_begin=5, sample_count=12)
    assert_same(batch(gpu_ctx, cams, seed=8, sample_begin=5, sample_count=12), part)
    # RT_B200_MAX_CHUNKS=1: at most 32 samples per launch, so 100 samples take 4 stream-ordered launches
    monkeypatch.setenv("RT_B200_MAX_CHUNKS", "1")
    small = rtb.Context(0)
    try:
        small.upload_scene(sc.desc)
        n0 = small.stats().kernel_launches
        cams100 = orbit(rtb, sc, 4, 40, 100)
        split = batch(small, cams100, seed=8)
        assert small.stats().kernel_launches - n0 >= 4  # 100 samples, <= 32 per launch
        assert_same(split, batch(gpu_ctx, cams100, seed=8))
    finally:
        small.close()


def test_downloads_and_state(rtb, gpu_ctx):
    sc = rtb.Scene("cornell_smoke", rand_seed=1)
    cams = orbit(rtb, sc, 3, 36, 10)
    gpu_ctx.upload_scene(sc.desc)
    per_view = []
    for cam in cams:
        gpu_ctx.render(cam, seed=6)
        assert gpu_ctx.stats().n_views == 1
        per_view.append((gpu_ctx.download_rgb8(10), gpu_ctx.download_radiance(10)))
    gpu_ctx.render_views(cams, seed=6)
    assert gpu_ctx.stats().n_views == 3
    rgb, rad = gpu_ctx.download_rgb8(10), gpu_ctx.download_radiance(10)
    H = rtb.image_height(cams[0])
    assert rgb.shape == rad.shape == (3, H, 36, 3)
    for v in range(3):
        assert np.array_equal(rgb[v], per_view[v][0]) and np.array_equal(rad[v], per_view[v][1])
    # the raw buffer is the whole batch, view-major
    ptr, nbytes = gpu_ctx.accum_ptr()
    assert nbytes == 3 * H * 36 * 3 * 8
    # V = 1 keeps the batch shape
    gpu_ctx.render_views(cams[:1], seed=6)
    assert gpu_ctx.stats().n_views == 1 and gpu_ctx.download_rgb8(10).shape == (1, H, 36, 3)
    assert np.array_equal(gpu_ctx.download_rgb8(10)[0], per_view[0][0])
    # a later render is single-image again, with its own bits, also with clear = 0 right after a batch
    gpu_ctx.render_views(cams, seed=6)
    gpu_ctx.render(cams[2], seed=6, clear=False)
    assert gpu_ctx.stats().n_views == 1
    img = gpu_ctx.download_rgb8(10)
    assert img.shape == (H, 36, 3) and np.array_equal(img, per_view[2][0])
    # and upload_accum too
    gpu_ctx.render_views(cams, seed=6)
    sums = gpu_ctx.download_accum()
    gpu_ctx.upload_accum(cams[1], sums[1])
    assert gpu_ctx.stats().n_views == 1
    assert np.array_equal(gpu_ctx.download_accum(), sums[1])


def test_refusals(rtb, gpu_ctx):
    lib = rtb.cuda_lib()
    sc = rtb.Scene("quads", rand_seed=1)
    cams = orbit(rtb, sc, 3, 32, 4)
    fresh = rtb.Context(0)
    try:
        with pytest.raises(rtb.RtError, match=r"\(-3\)"):
            fresh.render_views(cams)
    finally:
        fresh.close()
    gpu_ctx.upload_scene(sc.desc)

    def rc(cs, n=None, opts=None, arr=True):
        a = (rtb.rt_camera_desc * max(len(cs), 1))(*cs)
        o = opts or rtb.rt_render_opts(0, 0, 0, 1, 0, None, None)
        return lib.rt_render_views(gpu_ctx._h, len(cs) if n is None else n, a if arr else None, C.byref(o))

    assert rc([]) == rtb.RT_ERR_INVALID
    assert rc(cams, n=-1) == rtb.RT_ERR_INVALID
    assert rc(cams, arr=False) == rtb.RT_ERR_INVALID
    for field, value in (("image_width", 0), ("samples_per_pixel", 0), ("aspect_ratio", 0.0), ("aspect_ratio", float("nan"))):
        bad = orbit(rtb, sc, 3, 32, 4)
        setattr(bad[1], field, value)
        assert rc(bad) == rtb.RT_ERR_INVALID, field
    for field, value in (("image_width", 33), ("samples_per_pixel", 5), ("aspect_ratio", 2.0)):
        bad = orbit(rtb, sc, 3, 32, 4)
        setattr(bad[2], field, value)
        assert rc(bad) == rtb.RT_ERR_INVALID, field
    same_height = orbit(rtb, sc, 2, 32, 4)
    same_height[1].aspect_ratio = same_height[0].aspect_ratio * 0.999  # another ratio, the same int(W / ratio)
    assert rtb.image_height(same_height[0]) == rtb.image_height(same_height[1])
    assert rc(same_height) == rtb.RT_OK
    huge = orbit(rtb, sc, 2, 32768, 4)
    for c in huge:
        c.aspect_ratio = 0.5  # 32768 x 65536 = 2^31 pixels per view
    assert rc(huge) == rtb.RT_ERR_INVALID and rc(huge[:1]) == rtb.RT_ERR_INVALID
    assert rc(cams, opts=rtb.rt_render_opts(0, 4, 0, 1, 0, None, None)) == rtb.RT_ERR_INVALID  # empty sample range
    ptr, _ = gpu_ctx.accum_ptr()
    assert rc(cams, opts=rtb.rt_render_opts(0, 0, 0, 1, 0, ptr, None)) == rtb.RT_ERR_UNSUPPORTED
    assert rc(cams, opts=rtb.rt_render_opts(0, 0, 0, 1, 0, None, ptr)) == rtb.RT_ERR_UNSUPPORTED
    for flag in (rtb.RT_RENDER_COUNTERS, rtb.RT_RENDER_STREAM, rtb.RT_RENDER_REFILL):
        assert rc(cams, opts=rtb.rt_render_opts(0, 0, 0, 1, flag, None, None)) == rtb.RT_ERR_UNSUPPORTED, flag
    assert rc(cams, opts=rtb.rt_render_opts(0, 0, 0, 1, rtb.RT_RENDER_MEGAKERNEL, None, None)) == rtb.RT_OK
    gpu_ctx.synchronize()


def test_cpp_render_views_writes_what_camera_render_writes(rtb, tmp_path):
    """tests/cpp/views_main.cpp, built like the drop-in test builds its program: N frames through rtb200::render_views
    give the files and the stdout of N camera::render calls, on one context and sharded by views over three."""
    host = os.path.join(rtb.REPO_ROOT, "raytracing-practice_b200", "host")
    exe = str(tmp_path / "views")
    libdir = os.path.dirname(rtb.CUDA_LIB_PATH)
    cmd = ["g++", "-std=c++11", "-O1", "-I", host, "-I", os.path.join(rtb.REPO_ROOT, "include"),
           os.path.join(rtb.REPO_ROOT, "tests", "cpp", "views_main.cpp"), "-L", libdir, "-lrt_b200", "-Wl,-rpath," + libdir, "-o", exe]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    frames = 5

    def run(mode, devices):
        prefix = str(tmp_path / f"{mode}_{len(devices)}")
        r = subprocess.run([exe, "bouncing_spheres", prefix, "60", "12", str(frames), mode], capture_output=True, text=True,
                           env=dict(os.environ, RT_B200_DEVICES=devices))
        assert r.returncode == 0, r.stderr[-2000:]
        return [open(f"{prefix}_{i:03d}.ppm", "rb").read() for i in range(frames)], r.stdout

    loop, loop_out = run("loop", "0")
    assert loop_out.count("Done.") == frames
    assert len(set(loop)) == frames  # the frames differ
    for devices in ("0", "0,0,0"):
        files, out = run("batch", devices)
        assert out == loop_out
        for i in range(frames):
            assert files[i] == loop[i], (devices, i)
