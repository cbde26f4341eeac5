"""Build rt_scene_desc (include/rt_b200.h) directly from Python, for tests that need scenes the
named builders do not provide (random primitives, single features, malformed graphs).
Containers are plain lists (no bvh_node), so bounding boxes are not needed by the oracle."""
import ctypes as C
import importlib
import math

import numpy as np

abi = importlib.import_module("raytracing-practice_b200._abi")


class SceneDesc:
    def __init__(self):
        self.h, self.children, self.m, self.t, self.images, self.perlins = [], [], [], [], [], []
        self._keep = []
        self.n_prims = 0
        self.root = -1

    # ---- textures / materials -------------------------------------------------------------
    def _tex(self, kind, color=(0, 0, 0), scale=0.0, even=-1, odd=-1, image=-1, perlin=-1):
        t = abi.rt_texture(kind, even, odd, image, perlin, 0, (C.c_double * 3)(*color), scale)
        self.t.append(t)
        return len(self.t) - 1

    def solid(self, r, g, b):
        return self._tex(abi.RT_T_SOLID, (r, g, b))

    def checker(self, scale, even, odd):
        return self._tex(abi.RT_T_CHECKER, scale=1.0 / scale, even=even, odd=odd)

    def image(self, rgb8):
        """rgb8: HxWx3 uint8 array (already 'convert_to_bytes'-ed), or None for a failed load."""
        im = abi.rt_image()
        if rgb8 is None:
            im.width = im.height = 0
            im.rgb = None
        else:
            arr = np.ascontiguousarray(rgb8, np.uint8)
            self._keep.append(arr)
            im.height, im.width = arr.shape[:2]
            im.rgb = arr.ctypes.data_as(C.POINTER(C.c_uint8))
        self.images.append(im)
        return self._tex(abi.RT_T_IMAGE, image=len(self.images) - 1)

    def noise(self, scale, rng):
        p = abi.rt_perlin()
        v = rng.uniform(-1, 1, (256, 3))
        v /= np.linalg.norm(v, axis=1, keepdims=True)
        for i in range(256):
            for c in range(3):
                p.randvec[i][c] = v[i, c]
        for name in ("perm_x", "perm_y", "perm_z"):
            perm = rng.permutation(256)
            arr = getattr(p, name)
            for i in range(256):
                arr[i] = int(perm[i])
        self.perlins.append(p)
        return self._tex(abi.RT_T_NOISE, scale=scale, perlin=len(self.perlins) - 1)

    def _mat(self, kind, texture=-1, albedo=(0, 0, 0), fuzz=0.0, ior=0.0):
        self.m.append(abi.rt_material(kind, texture, (C.c_double * 3)(*albedo), fuzz, ior))
        return len(self.m) - 1

    def lambertian(self, tex):
        return self._mat(abi.RT_M_LAMBERTIAN, tex)

    def metal(self, albedo, fuzz):
        return self._mat(abi.RT_M_METAL, albedo=albedo, fuzz=min(fuzz, 1.0))

    def dielectric(self, ior):
        return self._mat(abi.RT_M_DIELECTRIC, ior=ior)

    def light(self, tex):
        return self._mat(abi.RT_M_DIFFUSE_LIGHT, tex)

    def isotropic(self, tex):
        return self._mat(abi.RT_M_ISOTROPIC, tex)

    # ---- hittables ------------------------------------------------------------------------
    def _hit(self, kind, material=-1, child0=-1, child1=-1, p=(), prim=False):
        h = abi.rt_hittable()
        h.kind, h.material, h.child0, h.child1 = kind, material, child0, child1
        h.prim_id = -1
        if prim:
            h.prim_id = self.n_prims
            self.n_prims += 1
        for i, v in enumerate(p):
            h.p[i] = v
        self.h.append(h)
        return len(self.h) - 1

    def sphere(self, c, r, mat, c2=None):
        d = (0, 0, 0) if c2 is None else tuple(np.float64(c2[i]) - np.float64(c[i]) for i in range(3))
        return self._hit(abi.RT_H_SPHERE, mat, p=(*c, *d, r), prim=True)

    def quad(self, q, u, v, mat):
        return self._hit(abi.RT_H_QUAD, mat, p=(*q, *u, *v), prim=True)

    def list(self, kids):
        first = len(self.children)
        self.children.extend(kids)
        return self._hit(abi.RT_H_LIST, child0=first, child1=len(kids))

    def box(self, a, b, mat):  # quad.hpp:129-159 order: +z, +x, -z, -x, +y, -y
        lo = [min(a[i], b[i]) for i in range(3)]
        hi = [max(a[i], b[i]) for i in range(3)]
        dx, dy, dz = (hi[0] - lo[0], 0, 0), (0, hi[1] - lo[1], 0), (0, 0, hi[2] - lo[2])
        neg = lambda v: tuple(-x for x in v)  # noqa: E731
        kids = [self.quad((lo[0], lo[1], hi[2]), dx, dy, mat), self.quad((hi[0], lo[1], hi[2]), neg(dz), dy, mat),
                self.quad((hi[0], lo[1], lo[2]), neg(dx), dy, mat), self.quad((lo[0], lo[1], lo[2]), dz, dy, mat),
                self.quad((lo[0], hi[1], hi[2]), dx, neg(dz), mat), self.quad((lo[0], lo[1], lo[2]), dx, dz, mat)]
        return self.list(kids)

    def translate(self, child, off):
        return self._hit(abi.RT_H_TRANSLATE, child0=child, p=off)

    def rotate_y(self, child, deg):
        rad = deg * 3.1415926535897932385 / 180.0
        return self._hit(abi.RT_H_ROTATE_Y, child0=child, p=(deg, math.sin(rad), math.cos(rad)))

    def medium(self, boundary, density, phase_mat):
        return self._hit(abi.RT_H_MEDIUM, phase_mat, child0=boundary, p=(density, -1 / density))

    # ---- finish ---------------------------------------------------------------------------
    def finish(self, root):
        self.root = root
        d = abi.rt_scene_desc()
        d.abi_version = abi.RT_B200_ABI_VERSION
        d.root = root
        arrays = [("hittables", self.h, abi.rt_hittable, "n_hittables"), ("materials", self.m, abi.rt_material, "n_materials"),
                  ("textures", self.t, abi.rt_texture, "n_textures"), ("images", self.images, abi.rt_image, "n_images"),
                  ("perlins", self.perlins, abi.rt_perlin, "n_perlins")]
        for field, items, typ, count in arrays:
            arr = (typ * max(len(items), 1))(*items)
            self._keep.append(arr)
            setattr(d, field, C.cast(arr, C.POINTER(typ)))
            setattr(d, count, len(items))
        ci = (C.c_int32 * max(len(self.children), 1))(*self.children)
        self._keep.append(ci)
        d.child_index = C.cast(ci, C.POINTER(C.c_int32))
        d.n_child_index = len(self.children)
        d.n_prims = self.n_prims
        self.desc = d
        return C.pointer(d)


def camera(width=64, aspect=1.0, spp=16, depth=10, bg=(0.7, 0.8, 1.0), vfov=40.0, lookfrom=(0, 0, 10), lookat=(0, 0, 0),
           vup=(0, 1, 0), defocus=0.0, focus=10.0):
    c = abi.rt_camera_desc()
    c.aspect_ratio, c.image_width, c.samples_per_pixel, c.max_depth = aspect, width, spp, depth
    c.vfov, c.defocus_angle, c.focus_dist = vfov, defocus, focus
    for i in range(3):
        c.background[i], c.lookfrom[i], c.lookat[i], c.vup[i] = bg[i], lookfrom[i], lookat[i], vup[i]
    return c


def random_scene(rng, n_spheres=40, n_quads=40, n_boxes=6):
    """Random spheres (40 % moving), quads and boxes under rotate_y + translate (half of them in nested wrappers), plus
    an instanced group of moving spheres: (SceneDesc, desc)."""
    s = SceneDesc()
    mat = s.lambertian(s.solid(0.5, 0.5, 0.5))
    kids = []
    for _ in range(n_spheres):
        c = rng.uniform(-10, 10, 3)
        c2 = c + rng.uniform(-1, 1, 3) if rng.random() < 0.4 else None
        kids.append(s.sphere(tuple(c), float(rng.uniform(0.2, 2.5)), mat, None if c2 is None else tuple(c2)))
    for _ in range(n_quads):
        kids.append(s.quad(tuple(rng.uniform(-10, 10, 3)), tuple(rng.uniform(-4, 4, 3)), tuple(rng.uniform(-4, 4, 3)), mat))
    for _ in range(n_boxes):
        b = s.box(tuple(rng.uniform(-2, 0, 3)), tuple(rng.uniform(0.5, 3, 3)), mat)
        b = s.rotate_y(b, float(rng.uniform(-80, 80)))
        b = s.translate(b, tuple(rng.uniform(-8, 8, 3)))
        if rng.random() < 0.5:  # nested wrappers
            b = s.translate(s.rotate_y(b, float(rng.uniform(-30, 30))), tuple(rng.uniform(-2, 2, 3)))
        kids.append(b)
    # instanced moving spheres
    sub = s.list([s.sphere(tuple(rng.uniform(-1, 1, 3)), 0.5, mat, tuple(rng.uniform(-1, 1, 3))) for _ in range(5)])
    kids.append(s.translate(s.rotate_y(sub, 33.0), (3.0, -2.0, 1.0)))
    return s, s.finish(s.list(kids))


def random_rays(rng, n):
    o = rng.uniform(-14, 14, (n, 3))
    target = rng.uniform(-9, 9, (n, 3))
    d = (target - o) * rng.uniform(0.05, 3.0, (n, 1))  # un-normalised, like the reference's rays
    return o, d, rng.uniform(0, 1, n)
