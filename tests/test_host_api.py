"""Host side of the boundary (no GPU): the C++ mirror of the reference's scene API, the
flattener, the JPEG decoder, and the scene converter inside the C-ABI library."""
import ctypes as C
import hashlib
import os
import subprocess

import numpy as np
import pytest

from conftest import ALL_SCENES

REF = os.environ.get("RT_B200_REFERENCE", "")  # a checkout of the reference project (its src/main.cpp)


def test_all_named_scenes_flatten(rtb, built, pins):
    assert set(rtb.scene_names()) == set(ALL_SCENES)
    for name in ALL_SCENES:
        sc = rtb.Scene(name, rand_seed=1)
        d = sc.desc.contents
        assert d.abi_version == rtb.RT_B200_ABI_VERSION and 0 <= d.root < d.n_hittables
        assert d.n_prims == pins["scenes"][name]["primary_full"]["prims"]
        kinds = [d.hittables[i].kind for i in range(d.n_hittables)]
        ids = sorted(d.hittables[i].prim_id for i in range(d.n_hittables) if kinds[i] in (rtb.RT_H_SPHERE, rtb.RT_H_QUAD))
        assert ids == list(range(d.n_prims))  # dense DFS numbering, shared leaves once
    d = rtb.Scene("book2_final", rand_seed=1).desc.contents
    kinds = [d.hittables[i].kind for i in range(d.n_hittables)]
    assert kinds.count(rtb.RT_H_MEDIUM) == 2 and kinds.count(rtb.RT_H_ROTATE_Y) == 1 and kinds.count(rtb.RT_H_TRANSLATE) == 1
    assert kinds.count(rtb.RT_H_QUAD) == 2401 and kinds.count(rtb.RT_H_SPHERE) == 1007
    assert d.n_perlins == 1 and d.n_images == 1


def test_scene_construction_follows_the_rand_stream(rtb, built):
    """rand() consumption: same seed -> identical bytes; the unseeded default is srand(1)."""
    a = rtb.Scene("bouncing_spheres", rand_seed=1)
    b = rtb.Scene("bouncing_spheres", rand_seed=1)
    c = rtb.Scene("bouncing_spheres", rand_seed=2)
    n = a.desc.contents.n_hittables
    raw = lambda s: C.string_at(s.desc.contents.hittables, n * C.sizeof(rtb.rt_hittable))  # noqa: E731
    assert raw(a) == raw(b) and a.desc.contents.n_hittables == b.desc.contents.n_hittables
    assert c.desc.contents.n_hittables != n or raw(c) != raw(a)


def test_jpeg_decoder_matches_libjpeg_bit_for_bit(rtb, built, earthmap):
    """The earth scenes' texture (the reference's earthmap.jpg or the stand-in, conftest.py) decodes to the texels libjpeg-turbo gives."""
    lib = rtb.scenes_lib()
    p, w, h = C.POINTER(C.c_uint8)(), C.c_int(), C.c_int()
    path = os.path.join(earthmap["dir"], "earthmap.jpg").encode()
    assert hashlib.sha256(open(path, "rb").read()).hexdigest() == earthmap["jpeg_sha256"]
    assert lib.rth_load_texture(path, 0, C.byref(p), C.byref(w), C.byref(h)) == 0
    assert (w.value, h.value) == (earthmap["width"], earthmap["height"])
    raw = C.string_at(p, w.value * h.value * 3)
    lib.rth_free(p)
    assert hashlib.sha256(raw).hexdigest() == earthmap["rgb8_sha256"]  # == PIL / libjpeg-turbo
    # rtw_image conventions on top: stb's gamma-2.2 linearisation then float_to_byte (SURVEY §8(c))
    assert lib.rth_load_texture(path, 1, C.byref(p), C.byref(w), C.byref(h)) == 0
    lin = np.frombuffer(C.string_at(p, w.value * h.value * 3), np.uint8)
    lib.rth_free(p)
    src = np.frombuffer(raw, np.uint8)
    lut = {64: 12, 128: 56, 200: 150, 254: 253, 255: 255, 0: 0}
    for k, v in lut.items():
        if (src == k).any():
            assert np.all(lin[src == k] == v)
    assert lib.rth_load_texture(b"/nonexistent/x.jpg", 0, C.byref(p), C.byref(w), C.byref(h)) != 0


def test_jpeg_decoder_subsampled_and_restart_files(rtb, built, tmp_path):
    """4:2:2 / 4:2:0 / grayscale / restart-interval files, encoded here with PIL, decoded by both."""
    Image = pytest.importorskip("PIL.Image")
    rng = np.random.default_rng(0)
    base = (rng.random((61, 83, 3)) * 255).astype(np.uint8)
    base = np.asarray(Image.fromarray(base).resize((83 * 2, 61 * 2), Image.BICUBIC))
    lib = rtb.scenes_lib()
    for tag, kw, mode in [("444", dict(subsampling=0), "RGB"), ("422", dict(subsampling=1), "RGB"), ("420", dict(subsampling=2), "RGB"),
                          ("gray", {}, "L"), ("rst", dict(subsampling=2, restart_marker_blocks=3), "RGB")]:
        path = str(tmp_path / f"{tag}.jpg")
        Image.fromarray(base).convert(mode).save(path, quality=88, **kw)
        want = np.asarray(Image.open(path).convert("RGB"))
        p, w, h = C.POINTER(C.c_uint8)(), C.c_int(), C.c_int()
        assert lib.rth_load_texture(path.encode(), 0, C.byref(p), C.byref(w), C.byref(h)) == 0, tag
        got = np.frombuffer(C.string_at(p, w.value * h.value * 3), np.uint8).reshape(h.value, w.value, 3)
        lib.rth_free(p)
        assert np.array_equal(got, want), tag


def test_jpeg_decoder_rejects_malformed_huffman_tables(rtb, built, tmp_path):
    """A crafted DHT whose code-length counts over-subscribe the code space (bits[1] = 200, stb_image rejects it too) must
    be refused by read_dht's Kraft check — before the fix the canonical-code loop wrote past the 512-entry lookup table —
    and truncated / garbage files must fail cleanly: rtw_image then falls back to its cyan texel (rtw_stb_image.hpp)."""
    Image = pytest.importorskip("PIL.Image")
    path = str(tmp_path / "ok.jpg")
    Image.fromarray((np.random.default_rng(1).random((16, 16, 3)) * 255).astype(np.uint8)).save(path, quality=80)
    data = bytearray(open(path, "rb").read())
    i = data.find(b"\xff\xc4")  # the first DHT segment: marker, length (2), Tc/Th (1), 16 counts
    assert i > 0
    lib = rtb.scenes_lib()
    p, w, h = C.POINTER(C.c_uint8)(), C.c_int(), C.c_int()
    for tag, mutate in [("oversubscribed", lambda d: d.__setitem__(i + 5, 200)), ("all_ones", lambda d: d.__setitem__(slice(i + 5, i + 21), bytes([255] * 16))),
                        ("truncated", lambda d: d.__delitem__(slice(len(d) // 2, len(d)))), ("garbage", lambda d: d.__setitem__(slice(2, 40), bytes(range(38))))]:
        d = bytearray(data)
        mutate(d)
        bad = str(tmp_path / f"{tag}.jpg")
        open(bad, "wb").write(bytes(d))
        rc = lib.rth_load_texture(bad.encode(), 0, C.byref(p), C.byref(w), C.byref(h))
        if tag in ("oversubscribed", "all_ones", "garbage"):
            assert rc != 0, tag  # refused, no crash
        elif rc == 0:  # a truncated scan may still decode (missing data reads as zero bits): must not crash, size intact
            assert (w.value, h.value) == (16, 16)
            lib.rth_free(p)
    assert lib.rth_load_texture(path.encode(), 0, C.byref(p), C.byref(w), C.byref(h)) == 0
    lib.rth_free(p)


def test_scene_converter_counts_and_errors(rtb, built):
    lib = C.CDLL(rtb.CUDA_LIB_PATH)
    lib.rt_debug_build_stats.argtypes = [C.POINTER(rtb.rt_scene_desc), C.POINTER(C.c_int32), C.POINTER(C.c_double)]
    # spheres, quad records, media, box() lists recognised as one slab-test primitive (quad.hpp:129-159)
    want = {"bouncing_spheres": (484, 0, 0, 0), "cornell_box": (0, 18, 0, 2), "cornell_smoke": (0, 18, 2, 2), "book2_final": (1008, 2401, 2, 400)}
    for name, (ns, nq, nm, nb) in want.items():
        sc = rtb.Scene(name, rand_seed=1)
        cnt = (C.c_int32 * 16)()
        assert lib.rt_debug_build_stats(sc.desc, cnt, None) == 0
        assert (cnt[1], cnt[2], cnt[3], cnt[8]) == (ns, nq, nm, nb), name
        assert 1 <= cnt[0] <= max(1, ns + nq) and cnt[5] <= 32  # nodes, depth within the traversal stack
    import scene_util as su

    s = su.SceneDesc()
    k = s.sphere((0, 0, 0), 1, s.lambertian(s.solid(1, 1, 1)))
    s.h[k].kind = 42
    assert lib.rt_debug_build_stats(s.finish(k), None, None) != 0
    s = su.SceneDesc()
    bad = s.finish(s.list([]))
    s.desc.root = 99
    assert lib.rt_debug_build_stats(bad, None, None) != 0


@pytest.mark.skipif(not os.path.isfile(os.path.join(REF, "src", "main.cpp")),
                    reason="needs the reference project's src/main.cpp, third-party source this repository does not hold: set RT_B200_REFERENCE "
                           "to a checkout of the reference")
def test_reference_main_cpp_compiles_unchanged_against_the_host_api(rtb, tmp_path):
    """Drop-in: the reference's own src/main.cpp (all seven scene functions + main) compiles against
    raytracing-practice_b200/host with no source change and links against the C-ABI library."""
    host = os.path.join(rtb.REPO_ROOT, "raytracing-practice_b200", "host")
    exe = str(tmp_path / "raytracer")
    # main.cpp is fed through stdin so that its quoted includes ("common/rtweekend.hpp", ...) resolve
    # through -I (our host API) instead of the reference's own directory; the text is untouched.
    cmd = ["g++", "-std=c++11", "-O1", "-x", "c++", "-", "-I", host, "-I", os.path.join(rtb.REPO_ROOT, "include"),
           "-L", os.path.dirname(rtb.CUDA_LIB_PATH), "-lrt_b200", "-Wl,-rpath," + os.path.dirname(rtb.CUDA_LIB_PATH), "-o", exe]
    r = subprocess.run(cmd, capture_output=True, text=True, cwd=str(tmp_path), input=open(os.path.join(REF, "src", "main.cpp"), encoding="utf-8").read())
    assert r.returncode == 0, r.stderr[-3000:]
    # without a GPU the binary must fail loudly (no CPU fallback), not render something else
    import torch

    if not torch.cuda.is_available():
        out = subprocess.run([exe, str(tmp_path / "image.ppm")], capture_output=True, text=True, cwd=str(tmp_path))
        assert out.returncode != 0 and "rt_init" in out.stderr


def test_box_lists_are_recognised_only_when_they_are_boxes(rtb, built):
    """The flattener turns a hittable_list into ONE slab-test primitive only if it is what box() builds
    (quad.hpp:129-159): six axis-aligned rectangles of one material tiling the surface of [lo, hi] — corners that are
    min + (max - min) may differ from max in the last bit.  Anything else stays six quads."""
    import numpy as np
    import scene_util as su

    lib = C.CDLL(rtb.CUDA_LIB_PATH)
    lib.rt_debug_build_stats.argtypes = [C.POINTER(rtb.rt_scene_desc), C.POINTER(C.c_int32), C.POINTER(C.c_double)]

    def boxes_of(build):
        s = su.SceneDesc()
        mat = s.lambertian(s.solid(0.5, 0.5, 0.5))
        root = build(s, mat)
        cnt = (C.c_int32 * 16)()
        assert lib.rt_debug_build_stats(s.finish(root), cnt, None) == 0
        return cnt[8], cnt[2]

    rng = np.random.default_rng(0)
    for _ in range(50):  # awkward doubles: lo + (hi - lo) != hi for many of these
        a, b = tuple(rng.uniform(-3, 0, 3) * np.pi), tuple(rng.uniform(0.1, 7, 3) / 3.0)
        assert boxes_of(lambda s, m: s.box(a, b, m)) == (1, 6)
    # instanced: translate(rotate_y(box)) is still one primitive
    assert boxes_of(lambda s, m: s.translate(s.rotate_y(s.box((0, 0, 0), (1, 2, 3), m), 33.0), (4, 5, 6))) == (1, 6)
    # two boxes in one list of 12 quads are not "a box"
    assert boxes_of(lambda s, m: s.list(s.children[s.h[s.box((0, 0, 0), (1, 1, 1), m)].child0:][:6] + s.children[s.h[s.box((2, 0, 0), (3, 1, 1), m)].child0:][:6]))[0] == 0

    def open_box(s, m):  # five faces + a lid that does not span the face
        k = s.box((0, 0, 0), (1, 1, 1), m)
        kids = s.children[s.h[k].child0:s.h[k].child0 + 6]
        kids[4] = s.quad((0, 1, 1), (0.5, 0, 0), (0, 0, -1), m)
        return s.list(kids)

    assert boxes_of(open_box)[0] == 0

    def two_materials(s, m):
        k = s.box((0, 0, 0), (1, 1, 1), m)
        kids = s.children[s.h[k].child0:s.h[k].child0 + 6]
        s.h[kids[2]].material = s.lambertian(s.solid(1, 0, 0))
        return s.list(kids)

    assert boxes_of(two_materials)[0] == 0
    # a sheared "box" (parallelogram faces) is not axis-aligned
    assert boxes_of(lambda s, m: s.list([s.quad((0, 0, 0), (1, 0.2, 0), (0, 1, 0), m) for _ in range(6)]))[0] == 0


def test_checkpoint_file_helpers(rtb, tmp_path):
    """RT_B200_CHECKPOINT's file layer on the CPU: round trip, replacement, refusal of another render's file, and the
    scene hash telling two cameras / scenes apart (the GPU side is tests/test_gpu_render.py::test_cpp_checkpointed_*)."""
    import os
    import subprocess

    host = os.path.join(rtb.REPO_ROOT, "raytracing-practice_b200", "host")
    libdir = os.path.dirname(rtb.CUDA_LIB_PATH)
    exe = str(tmp_path / "ckpt_unit")
    r = subprocess.run(["g++", "-std=c++11", "-O1", "-Wall", "-I", host, "-I", os.path.join(rtb.REPO_ROOT, "include"),
                        os.path.join(rtb.REPO_ROOT, "tests", "cpp", "ckpt_unit.cpp"), "-L", libdir, "-lrt_b200", "-Wl,-rpath," + libdir, "-o", exe],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    ck = str(tmp_path / "a.ckpt")
    r = subprocess.run([exe, ck, "roundtrip"], capture_output=True, text=True)
    assert r.returncode == 0, (r.returncode, r.stderr)
    assert os.path.getsize(ck) == 48 + 5 * 3 * 3 * 8 and not os.path.exists(ck + ".tmp")
    for mode in ("other_scene", "other_spp"):
        r = subprocess.run([exe, ck, mode], capture_output=True, text=True)
        assert r.returncode == 1 and "another scene, camera or sample count" in r.stderr
    with open(ck, "r+b") as f:  # a truncated file is refused too
        f.truncate(100)
    r = subprocess.run([exe, ck, "same"], capture_output=True, text=True)
    assert r.returncode == 1 and "truncated" in r.stderr
