"""Generate the stand-in for the reference's images/earthmap.jpg and its pins.

The reference's texture asset is not part of this repository, and without it the two scenes that use it ("earth",
"book2_final") fall back to rtw_image's constant cyan texel.  Unless RTW_IMAGES holds the reference's image (then the
tests use ref_pins.json's "earthmap" entry and P3 pins), tests/conftest.py points RTW_IMAGES at tests/golden/images:

  * images/earthmap.jpg   : a seeded, earth-like 1024x512 equirectangular map, baseline JPEG 4:2:0 (what PIL writes)
  * earthmap_standin.json : sha256 of the file; sha256 of the RGB8 texels PIL (libjpeg-turbo) decodes from it; and,
                            for every named scene with an image texture, sha256 of oracle/liboracle.so's camera::render
                            P3 text on the stand-in at the reduced size of ref_pins.json ("small") and, for the
                            shipped scenes tests/test_oracle_golden.py renders at full size, at that size ("shipped").

The P3 pins are outputs of the oracle, which reproduces the reference bit for bit on the real earthmap.jpg
(ref_pins.json); ray counts do not depend on texel values and stay pinned to the reference there.

    python tests/golden/make_standin.py            # after __graft_entry__.build(); rewrites both files
"""
import hashlib
import io
import json
import os
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
IMAGE_DIR = os.path.join(HERE, "images")
SHIPPED = ["earth", "checkered_spheres"]  # the shipped-size renders of tests/test_oracle_golden.py


def sha(b):
    return hashlib.sha256(b).hexdigest()


def standin_rgb8(width=1024, height=512, seed=20240601):
    """Oceans, continents and ice caps from smooth random fields on the sphere (seamless across the date line)."""
    rng = np.random.default_rng(seed)
    lat = (0.5 - (np.arange(height) + 0.5) / height) * np.pi
    lon = (np.arange(width) + 0.5) / width * 2.0 * np.pi
    lon, lat = np.meshgrid(lon, lat)
    p = np.stack([np.cos(lat) * np.cos(lon), np.cos(lat) * np.sin(lon), np.sin(lat)], axis=-1)

    def field(n, f_lo, f_hi):
        d = rng.normal(size=(n, 3))
        d /= np.linalg.norm(d, axis=1, keepdims=True)
        f = rng.uniform(f_lo, f_hi, n)
        ph = rng.uniform(0, 2 * np.pi, n)
        return sum(np.sin(f[k] * (p @ d[k]) + ph[k]) / np.sqrt(f[k]) for k in range(n)) / np.sqrt(n)

    land = np.clip((field(24, 1.5, 9.0) - 0.05) * 6.0, 0.0, 1.0)
    relief = 0.5 + 0.5 * np.tanh(2.0 * field(16, 3.0, 14.0) + 0.8 * field(48, 20.0, 90.0))
    depth = 0.5 + 0.5 * np.tanh(1.5 * field(32, 6.0, 60.0))
    ocean = np.array([0.04, 0.12, 0.36]) + 0.1 * depth[..., None] * np.array([0.0, 0.4, 0.5])
    ground = (1.0 - relief[..., None]) * np.array([0.16, 0.42, 0.12]) + relief[..., None] * np.array([0.55, 0.45, 0.28])
    ice = np.clip((np.abs(lat) - np.radians(66.0)) / np.radians(6.0), 0.0, 1.0)[..., None]
    rgb = land[..., None] * ground + (1.0 - land[..., None]) * ocean
    rgb = (1.0 - ice) * rgb + ice * np.array([0.92, 0.94, 0.96])
    return np.clip(np.rint(rgb * 255.0), 0, 255).astype(np.uint8)


def main():
    from PIL import Image

    os.makedirs(IMAGE_DIR, exist_ok=True)
    path = os.path.join(IMAGE_DIR, "earthmap.jpg")
    buf = io.BytesIO()
    Image.fromarray(standin_rgb8()).save(buf, format="JPEG", quality=75)
    open(path, "wb").write(buf.getvalue())
    decoded = np.asarray(Image.open(path).convert("RGB"))
    pins = {"jpeg_sha256": sha(buf.getvalue()), "rgb8_sha256": sha(decoded.tobytes()),
            "width": int(decoded.shape[1]), "height": int(decoded.shape[0]), "small": {}, "shipped": {}}

    os.environ["RTW_IMAGES"] = IMAGE_DIR
    sys.path.insert(0, ROOT)
    import importlib

    from oracle import orc

    rtb = importlib.import_module("raytracing-practice_b200")
    small = json.load(open(os.path.join(HERE, "ref_pins.json")))["small"]
    with tempfile.TemporaryDirectory() as tmp:
        out = os.path.join(tmp, "o.ppm")
        for name in rtb.scene_names():
            sc = rtb.Scene(name, rand_seed=1)
            if sc.desc.contents.n_images == 0:
                continue
            cam = sc.camera_copy(image_width=small["width"], samples_per_pixel=small["spp"], max_depth=small["depth"])
            orc.render_ppm(sc.desc, cam, out)
            pins["small"][name] = sha(open(out, "rb").read())
            if name in SHIPPED:
                sc = rtb.Scene(name, rand_seed=1)
                orc.render_ppm(sc.desc, sc.cam.contents, out)
                pins["shipped"][name] = sha(open(out, "rb").read())
            print(name, pins["small"][name][:16], pins["shipped"].get(name, "")[:16], flush=True)
    json.dump(pins, open(os.path.join(HERE, "earthmap_standin.json"), "w"), indent=1, sort_keys=True)
    print("wrote", path, f"({len(buf.getvalue())} bytes)")


if __name__ == "__main__":
    main()
