import hashlib
import importlib
import json
import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# The scenes with an image texture ("earth", "book2_final") load earthmap.jpg from RTW_IMAGES.  The reference's image is
# not part of this repository.  When RTW_IMAGES holds it (recognised by its sha256 in ref_pins.json), the tests compare
# with the reference's own pins; otherwise they read a generated stand-in of the same size and format
# (tests/golden/make_standin.py) and compare with the pins taken on it.  EARTHMAP holds whichever pins apply.
GOLDEN = os.path.join(ROOT, "tests", "golden")


def _earthmap_pins():
    ref = json.load(open(os.path.join(GOLDEN, "ref_pins.json")))
    d = os.environ.get("RTW_IMAGES", "")
    path = os.path.join(d, "earthmap.jpg")
    if d and os.path.isfile(path) and hashlib.sha256(open(path, "rb").read()).hexdigest() == ref["earthmap"]["jpeg_sha256"]:
        return dict(ref["earthmap"], dir=d, small={n: s["ppm"]["sha256"] for n, s in ref["scenes"].items()},
                    shipped={n: s["ppm_sha256"] for n, s in ref["shipped"].items()})
    return dict(json.load(open(os.path.join(GOLDEN, "earthmap_standin.json"))), dir=os.path.join(GOLDEN, "images"))


EARTHMAP = _earthmap_pins()
os.environ["RTW_IMAGES"] = EARTHMAP["dir"]


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")
    config.addinivalue_line("markers", "slow: long CPU oracle runs")


@pytest.fixture(scope="session")
def rtb():
    """The product package (directory name has a hyphen, hence importlib)."""
    return importlib.import_module("raytracing-practice_b200")


@pytest.fixture(scope="session")
def orc():
    """The CPU oracle binding — test infrastructure only."""
    from oracle import orc as o

    if not os.path.exists(o.LIB_PATH):
        import __graft_entry__ as g

        g.build()
    return o


@pytest.fixture(scope="session")
def pins():
    with open(os.path.join(ROOT, "tests", "golden", "ref_pins.json")) as f:
        return json.load(f)


@pytest.fixture(scope="session")
def earthmap():
    """Pins of the earthmap.jpg the tests render with: the reference's image when RTW_IMAGES holds it, else the stand-in."""
    return EARTHMAP


@pytest.fixture(scope="session")
def built(rtb):
    """Make sure the in-tree shared libraries exist (build() is a no-op when they are fresh)."""
    if not (os.path.exists(rtb.CUDA_LIB_PATH) and os.path.exists(rtb.SCENES_LIB_PATH)):
        import __graft_entry__ as g

        g.build()
    return True


@pytest.fixture(scope="session")
def gpu_ctx(rtb, built):
    ctx = rtb.Context(0)  # raises loudly when the CUDA library or the device is missing
    yield ctx
    ctx.close()


ALL_SCENES = ["bouncing_spheres", "checkered_spheres", "earth", "perlin_sphere", "quads", "simple_light", "cornell_box",
              "book1_final", "cornell_rotated", "cornell_smoke", "book2_final"]
