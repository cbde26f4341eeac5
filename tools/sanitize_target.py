"""The workload compute-sanitizer runs over (tools/sanitize.sh): every kernel of the library on small inputs —
smoke-sized parity queries, random-scene closest hits, 64-pixel renders of book2_final and cornell_smoke with every render
kernel (and the instrumented variants), a batch of views (rt_render_views), the push / adopt / peer paths with two contexts,
finalize + downloads.
Asserts the kernels still agree with each other, so a sanitizer-induced timing change cannot hide a race."""
import importlib, os, sys
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
rtb = importlib.import_module("raytracing-practice_b200")

WIDTH = int(os.environ.get("SAN_WIDTH", "64"))
SPP = int(os.environ.get("SAN_SPP", "4"))
ctx = rtb.Context(0)
rng = np.random.default_rng(3)
if os.environ.get("SAN_SELFTEST"):  # a checks build with RT_B200_CHECK_SELFTEST=1: the planted bad reference must be reported
    sc = rtb.Scene("bouncing_spheres", rand_seed=1)
    ctx.upload_scene(sc.desc)
    ctx.render(sc.camera_copy(image_width=64, samples_per_pixel=2, max_depth=8), seed=1)
    try:
        ctx.synchronize()
        print("SELFTEST: nothing reported")
    except rtb.RtError as e:
        print("SELFTEST:", e)
    sys.exit(0)
for name, depth in (("book2_final", 40), ("cornell_smoke", 50), ("bouncing_spheres", 20), ("perlin_sphere", 10), ("earth", 10), ("quads", 10)):
    sc = rtb.Scene(name, rand_seed=1)
    cam = sc.camera_copy(image_width=WIDTH, samples_per_pixel=SPP, max_depth=depth)
    ctx.upload_scene(sc.desc)
    # parity queries: exact, fp32, the render kernel's own instantiation
    ids = {}
    for tag, flags in (("exact", rtb.RT_TRACE_EXACT | rtb.RT_TRACE_SKIP_MEDIA), ("fp32", rtb.RT_TRACE_FP32 | rtb.RT_TRACE_SKIP_MEDIA),
                       ("render", rtb.RT_TRACE_RENDER_KERNEL | rtb.RT_TRACE_SKIP_MEDIA)):
        ids[tag] = ctx.primary_visibility(cam, flags)[0]
    assert (ids["render"] != ids["exact"]).mean() < 0.01
    n = 2000
    o = rng.uniform(-300, 600, (n, 3))
    d = rng.normal(size=(n, 3))
    ctx.trace_rays(o, d, rng.uniform(0, 1, n), 0.001, np.inf, rtb.RT_TRACE_FP32)
    ctx.trace_rays(o, d, None, 0.001, np.inf, rtb.RT_TRACE_EXACT)
    # bounce rays: the start-primitive rules of the fp32 traversal, and the render kernel's own second segment
    ids0 = ctx.primary_visibility(cam, rtb.RT_TRACE_EXACT | rtb.RT_TRACE_SKIP_MEDIA)[0].reshape(-1)
    starts = rng.choice(np.unique(ids0[ids0 >= 0]), n)
    ctx.trace_rays(o, d, rng.uniform(0, 1, n), 0.001, np.inf, rtb.RT_TRACE_FP32, start_prim=starts)
    b = ctx.bounce_visibility(cam, seed=9)
    assert (b["id"] == ids["render"]).all()
    # every render kernel, same bits
    acc = {}
    for tag, flags in (("mega", rtb.RT_RENDER_MEGAKERNEL), ("stream", rtb.RT_RENDER_STREAM), ("refill", rtb.RT_RENDER_REFILL),
                       ("mega+count", rtb.RT_RENDER_MEGAKERNEL | rtb.RT_RENDER_COUNTERS), ("refill+count", rtb.RT_RENDER_REFILL | rtb.RT_RENDER_COUNTERS)):
        try:
            ctx.render(cam, seed=9, flags=flags)
            acc[tag] = ctx.download_accum()
        except rtb.RtError as e:
            print(name, tag, "refused:", e)
    for tag, a in acc.items():
        assert np.array_equal(a, acc["mega"]), (name, tag)
    # a batch of views (render_kernel's VIEWS instantiation under this scene's plan): each view = its single render
    views = [sc.camera_copy(image_width=WIDTH, samples_per_pixel=SPP, max_depth=md, vfov=30.0 + 5 * i) for i, md in enumerate((depth, 3, 0))]
    ctx.render_views(views, seed=9)
    batch = ctx.download_accum()
    for i, v in enumerate(views):
        ctx.render(v, seed=9)
        assert np.array_equal(ctx.download_accum(), batch[i]), (name, "view", i)
    if os.environ.get("SAN_HASH"):
        import hashlib
        print("HASH", name, hashlib.sha1(acc["mega"].tobytes()).hexdigest()[:12], flush=True)
        print("HASH", name, "views", hashlib.sha1(batch.tobytes()).hexdigest()[:12], flush=True)
    ctx.download_rgb8(SPP), ctx.download_radiance(SPP), ctx.stats()
    ctx.synchronize()  # a checks build reports failed device-side checks here
    print(name, "ok:", sorted(acc), flush=True)
    if name == "cornell_smoke":  # the exchange step: push into a reduce buffer, adopt; and adds straight into a peer accumulator
        other = rtb.Context(0)
        other.upload_scene(sc.desc)
        ptr, handle = ctx.reduce_buffer(cam)
        ctx.render(cam, seed=9, sample_begin=0, sample_count=SPP // 2, push_accum=ptr)
        other.render(cam, seed=9, sample_begin=SPP // 2, sample_count=SPP - SPP // 2, push_accum=ptr)
        ctx.synchronize(), other.synchronize()
        ctx.adopt_reduce_buffer()
        assert np.array_equal(ctx.download_accum(), acc["mega"])
        ctx.render(cam, seed=9, sample_begin=0, sample_count=SPP // 2)
        ctx.synchronize()
        aptr, nbytes = ctx.accum_ptr()
        other.render(cam, seed=9, sample_begin=SPP // 2, sample_count=SPP - SPP // 2, peer_accum=aptr)
        other.synchronize()
        assert np.array_equal(ctx.download_accum(), acc["mega"])
        other.close()
        print("push / adopt / peer ok", flush=True)
    sc.close()
ctx.close()
print("sanitize target done")
