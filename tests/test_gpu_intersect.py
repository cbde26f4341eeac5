"""T1 — device intersection routines vs the oracle's sphere::hit / quad::hit / translate /
rotate_y on random rays over random scenes (fp64 exact predicate: bit-exact ids and t)."""
import numpy as np
import pytest

import scene_util as su

pytestmark = pytest.mark.gpu


random_scene, random_rays = su.random_scene, su.random_rays


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_exact_closest_hit_on_random_scenes(rtb, orc, gpu_ctx, seed):
    rng = np.random.default_rng(seed)
    s, desc = random_scene(rng)
    gpu_ctx.upload_scene(desc)
    o, d, tm = random_rays(rng, 200_000)
    for tmin, tmax in [(0.001, np.inf), (0.3, 1.1), (-np.inf, np.inf)]:
        ids, t, nrm, ff = gpu_ctx.trace_rays(o, d, tm, tmin, tmax, rtb.RT_TRACE_EXACT)
        oi, ot, on, of, _ = orc.hit_rays(desc, o, d, tm, tmin, tmax)
        assert np.array_equal(ids, oi)
        hit = oi >= 0
        assert hit.mean() > 0.2
        assert np.array_equal(t[hit], ot[hit])  # same operations in the same order: bit-identical
        assert np.array_equal(nrm[hit], on[hit])
        assert np.array_equal(ff[hit], of[hit])


def test_fp32_closest_hit_on_random_scenes(rtb, orc, gpu_ctx):
    rng = np.random.default_rng(7)
    s, desc = random_scene(rng)
    gpu_ctx.upload_scene(desc)
    o, d, tm = random_rays(rng, 200_000)
    ids, t, nrm, ff = gpu_ctx.trace_rays(o, d, tm, 0.001, np.inf, rtb.RT_TRACE_FP32)
    oi, ot, on, of, _ = orc.hit_rays(desc, o, d, tm, 0.001, np.inf)
    agree = ids == oi
    assert agree.mean() >= 0.999
    ok = agree & (oi >= 0)
    assert np.quantile(np.abs(t[ok] - ot[ok]) / np.abs(ot[ok]), 0.999) <= 1e-4
    assert np.array_equal(ff[ok], of[ok]) or (ff[ok] != of[ok]).mean() < 1e-4


def test_tie_rules_quads_inclusive_spheres_exclusive(rtb, orc, gpu_ctx):
    """SURVEY A.4/A.5: a later QUAD at exactly equal t replaces the earlier hit, a later SPHERE does not."""
    s = su.SceneDesc()
    mat = s.lambertian(s.solid(0.5, 0.5, 0.5))
    q0 = s.quad((-1, -1, 0), (2, 0, 0), (0, 2, 0), mat)
    q1 = s.quad((-1, -1, 0), (2, 0, 0), (0, 2, 0), mat)  # coincident, later in the list
    sp0 = s.sphere((5, 0, -1), 1.0, mat)
    sp1 = s.sphere((5, 0, -1), 1.0, mat)  # coincident spheres: the first one keeps the hit
    desc = s.finish(s.list([q0, q1, sp0, sp1]))
    gpu_ctx.upload_scene(desc)
    o = np.array([[0.25, 0.25, 4.0], [5.0, 0.0, 4.0]])
    d = np.array([[0.0, 0.0, -2.0], [0.0, 0.0, -2.0]])
    ids, t, _, _ = gpu_ctx.trace_rays(o, d, None, 0.001, np.inf, rtb.RT_TRACE_EXACT)
    oi, ot, *_ = orc.hit_rays(desc, o, d)
    assert list(oi) == [1, 2] and list(ids) == [1, 2]
    assert np.array_equal(t, ot)


def test_empty_and_single_primitive_worlds(rtb, orc, gpu_ctx):
    rng = np.random.default_rng(3)
    o, d, tm = random_rays(rng, 5000)
    s = su.SceneDesc()
    desc = s.finish(s.list([]))
    gpu_ctx.upload_scene(desc)
    for flags in (rtb.RT_TRACE_EXACT, rtb.RT_TRACE_FP32):
        ids, t, _, _ = gpu_ctx.trace_rays(o, d, tm, flags=flags)
        assert np.all(ids == -1) and np.all(np.isinf(t))
    s = su.SceneDesc()
    desc = s.finish(s.sphere((0, 0, 0), 6.0, s.lambertian(s.solid(1, 1, 1))))  # root is a bare primitive
    gpu_ctx.upload_scene(desc)
    ids, t, _, _ = gpu_ctx.trace_rays(o, d, tm, flags=rtb.RT_TRACE_EXACT)
    oi, ot, *_ = orc.hit_rays(desc, o, d, tm)
    assert np.array_equal(ids, oi) and np.array_equal(t[oi >= 0], ot[oi >= 0])
    ids, _, _, _ = gpu_ctx.trace_rays(o[:0], d[:0], tm[:0])  # zero rays
    assert ids.size == 0


def test_medium_boundary_spans(rtb, orc, gpu_ctx):
    """constant_medium's deterministic part: boundary entry/exit (rec1.t, rec2.t) within 1e-5 relative
    (SURVEY.md §8(c)); box boundaries under rotate_y+translate and sphere boundaries."""
    rng = np.random.default_rng(11)
    for name, n_media in (("cornell_smoke", 2), ("book2_final", 2)):
        sc = rtb.Scene(name, rand_seed=1)
        gpu_ctx.upload_scene(sc.desc)
        assert gpu_ctx.stats().n_media == n_media
        n = 100_000
        o = rng.uniform(-100, 655, (n, 3))
        target = rng.uniform(0, 555, (n, 3))
        d = (target - o) * rng.uniform(0.01, 2.0, (n, 1))
        for m in range(n_media):
            t1, t2 = gpu_ctx.medium_spans(m, o, d)
            o1, o2 = orc.medium_spans(sc.desc, m, o, d)
            both = ~np.isnan(o2) & ~np.isnan(t2)
            assert (np.isnan(o2) != np.isnan(t2)).mean() < 2e-3
            assert both.mean() > 0.05
            scale = np.maximum(np.abs(o2[both]), np.abs(o1[both]))
            assert np.quantile(np.abs(t1[both] - o1[both]) / scale, 0.999) <= 1e-5 * 10
            assert np.quantile(np.abs(t2[both] - o2[both]) / scale, 0.999) <= 1e-5 * 10
            assert np.median(np.abs(t2[both] - o2[both]) / scale) <= 1e-6


def test_large_scene_bvh_beyond_shared_memory(rtb, orc, gpu_ctx):
    """20,000 spheres + 300 instanced boxes: ~13 k BVH nodes = 0.85 MB, four times what fits in a CTA's shared
    memory, so the lower levels are fetched through L1/L2 (load_node's global branch) and the stacks run deep.
    Exact closest hit against the oracle's linear scan, the fp32 production traversal against the exact one,
    and both render kernels against each other."""
    rng = np.random.default_rng(21)
    s = su.SceneDesc()
    mat = s.lambertian(s.solid(0.6, 0.5, 0.4))
    kids = [s.sphere(tuple(rng.uniform(-40, 40, 3)), float(rng.uniform(0.1, 1.2)), mat) for _ in range(20_000)]
    for _ in range(300):
        b = s.box(tuple(rng.uniform(-1.5, 0, 3)), tuple(rng.uniform(0.3, 1.5, 3)), mat)
        kids.append(s.translate(s.rotate_y(b, float(rng.uniform(-90, 90))), tuple(rng.uniform(-40, 40, 3))))
    desc = s.finish(s.list(kids))
    gpu_ctx.upload_scene(desc)
    st = gpu_ctx.stats()
    assert st.n_boxes == 300 and st.n_nodes * 64 > 300_000 and st.bvh_nodes_in_smem < st.n_nodes
    n = 20_000
    o = rng.uniform(-45, 45, (n, 3))
    d = (rng.uniform(-40, 40, (n, 3)) - o) * rng.uniform(0.05, 2.0, (n, 1))
    ids, t, nrm, ff = gpu_ctx.trace_rays(o, d, None, 0.001, np.inf, rtb.RT_TRACE_EXACT)
    oi, ot, on, of, _ = orc.hit_rays(desc, o, d, None, 0.001, np.inf)
    assert np.array_equal(ids, oi) and (oi >= 0).mean() > 0.5
    hit = oi >= 0
    assert np.array_equal(t[hit], ot[hit]) and np.array_equal(nrm[hit], on[hit])
    ids32, t32, _, _ = gpu_ctx.trace_rays(o, d, None, 0.001, np.inf, rtb.RT_TRACE_FP32)
    assert (ids32 == oi).mean() >= 0.999
    cam = su.camera(width=160, spp=8, depth=6, lookfrom=(0, 0, 70), vfov=60.0)
    gpu_ctx.render(cam, seed=2, flags=rtb.RT_RENDER_MEGAKERNEL)
    a, r = gpu_ctx.download_accum(), gpu_ctx.stats().rays
    gpu_ctx.render(cam, seed=2, flags=rtb.RT_RENDER_REFILL)
    assert np.array_equal(a, gpu_ctx.download_accum()) and r == gpu_ctx.stats().rays and a.any()
