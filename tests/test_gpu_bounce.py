"""T2b — rays that start ON a surface, as every ray after the first of an rt_render path does, against the fp64 oracle.

A bounce ray avoids its own surface through a start-primitive rule, not an epsilon (rt_device.cuh: a sphere gets the
roots 0 and -2b/a, a quad is skipped, a box face's slab plane is crossed at exactly 0); the oracle (the reference) uses
interval(0.001, inf) instead.  The two must pick the same primitive:
  (a) the leaf rules on their own (rt_trace_rays_from): start points on adversarial features — the r = 1000 ground,
      r = 0.05 spheres, moving and nested spheres, coincident quads, rotated / nested boxes, their edges and corners,
      touching geometry — with outward, inward and near-tangent directions;
  (b) the render kernel's own second segment (rt_bounce_visibility) on every scene at full size and on three
      constructed ones, against the oracle's closest hit from the oracle's primary hit point along the kernel's d1;
  (c) one scene under every launch plan of the megakernel (BVH staged or not, stack in shared or local memory,
      cooperative turbulence, the instrumented kernel): the same bits.
Bounds are B200 measurements + 25 % (tools/bounce_parity.py -> profiles/r3_bounce_parity.md)."""
import contextlib
import math
import os

import numpy as np
import pytest

import scene_util as su
from conftest import ALL_SCENES

SCALE = 10.0  # extent of the adversarial scene: "interior" start points are >= 1e-4 * SCALE from every edge
EDGE_TYPES = ("quad_edge", "box_edge", "box_corner")
DIR_CLASSES = ("out", "in", "tangent")


def _unit(v):
    return v / np.linalg.norm(v, axis=-1, keepdims=True)


def _perp(rng, n):
    """A random unit vector perpendicular to each row of n."""
    r = rng.normal(size=n.shape)
    r -= np.sum(r * n, axis=1, keepdims=True) * n
    return _unit(r)


class _Xf:
    """Object -> world of nested rotate_y / translate wrappers, innermost first (oracle.cpp, RT_H_ROTATE_Y)."""

    def __init__(self, ops=()):
        self.ops = list(ops)

    def point(self, p, vec=False):
        p = np.array(p, np.float64)
        for kind, a in self.ops:
            if kind == "r":
                rad = a * 3.1415926535897932385 / 180.0
                sn, cs = math.sin(rad), math.cos(rad)
                x, z = p[..., 0].copy(), p[..., 2].copy()
                p[..., 0], p[..., 2] = cs * x + sn * z, -sn * x + cs * z
            elif not vec:
                p = p + np.array(a)
        return p

    def wrap(self, s, h):
        for kind, a in self.ops:
            h = s.rotate_y(h, a) if kind == "r" else s.translate(h, a)
        return h


def _box_ids(s, h):
    return [s.h[s.children[s.h[h].child0 + k]].prim_id for k in range(6)]


def adversarial_scene():
    """The scene of part (a) and, per start type, a sampler of (target point, outward aim, feature ids)."""
    s = su.SceneDesc()
    mat = s.lambertian(s.solid(0.5, 0.5, 0.5))
    glass = s.dielectric(1.5)
    kids, spheres, quads, boxes = [], [], [], []

    def sphere(kind, c, r, c2=None, m=mat):
        h = s.sphere(c, r, m, c2)
        kids.append(h)
        spheres.append((kind, np.array(c, np.float64), r, None if c2 is None else np.array(c2, np.float64) - np.array(c, np.float64), s.h[h].prim_id))

    sphere("ground", (0.0, -1000.0, 0.0), 1000.0)
    rng = np.random.default_rng(5)
    for x, z in rng.uniform(-7, 7, (12, 2)):
        sphere("small", (float(x), 0.05, float(z)), 0.05)  # resting on the ground: touching at (x, 0, z)
    for _ in range(5):
        c = rng.uniform(-6, 6, 3) + (0, 3, 0)
        sphere("moving", tuple(c), float(rng.uniform(0.3, 0.8)), tuple(c + rng.uniform(-1, 1, 3)))
    sphere("nested_outer", (-3.0, 2.0, 4.0), 1.2, m=glass)
    sphere("nested_inner", (-3.0, 2.0, 4.0), 0.8, m=glass)
    for i in range(8):
        q, u, v = rng.uniform(-8, 8, 3) + (0, 4, 0), rng.uniform(-3, 3, 3), rng.uniform(-3, 3, 3)
        h = s.quad(tuple(q), tuple(u), tuple(v), mat)
        kids.append(h)
        quads.append(("quad", q, u, v, [s.h[h].prim_id]))
    q, u, v = np.array([2.0, 6.0, -6.0]), np.array([2.0, 0.5, 0.0]), np.array([0.0, 0.3, 2.0])
    h0, h1 = s.quad(tuple(q), tuple(u), tuple(v), mat), s.quad(tuple(q), tuple(u), tuple(v), mat)  # coincident: the later one wins
    kids += [h0, h1]
    quads.append(("quad_coincident", q, u, v, [s.h[h0].prim_id, s.h[h1].prim_id]))
    for lo, hi, xf in [((-1.0, 0.0, -1.0), (0.5, 1.5, 0.8), _Xf([("t", (6.0, 0.0, 2.0))])),
                       ((-0.7, 0.0, -0.4), (0.9, 2.0, 0.6), _Xf([("r", 37.0), ("t", (-6.0, 0.0, -2.0))])),
                       ((-0.5, -0.5, -0.5), (0.5, 0.5, 0.5), _Xf([("r", -15.0), ("t", (0.3, 0.2, -0.1)), ("r", 52.0), ("t", (0.0, 3.5, -7.0))]))]:
        h = s.box(lo, hi, mat)
        ids = _box_ids(s, h)
        kids.append(xf.wrap(s, h))
        boxes.append(("box", np.array(lo), np.array(hi), xf, ids))
    # two boxes stacked face to face, rotated together
    xf = _Xf([("r", 30.0), ("t", (2.0, 0.0, 6.0))])
    a, b = s.box((-1.0, 0.0, -1.0), (1.0, 1.0, 1.0), mat), s.box((-0.5, 1.0, -0.5), (0.5, 2.0, 0.5), mat)
    kids.append(xf.wrap(s, s.list([a, b])))
    stack = [(np.array((-1.0, 0.0, -1.0)), np.array((1.0, 1.0, 1.0)), xf, _box_ids(s, a)),
             (np.array((-0.5, 1.0, -0.5)), np.array((0.5, 2.0, 0.5)), xf, _box_ids(s, b))]
    desc = s.finish(s.list(kids))
    return s, desc, dict(spheres=spheres, quads=quads, boxes=boxes, stack=stack)


def _aim_sphere(rng, c, r, dc, n, u_filter=None, inside=False):
    tm = rng.uniform(0, 1, n)
    cen = c + (tm[:, None] * dc if dc is not None else 0.0)
    u = _unit(rng.normal(size=(n, 3)))
    if u_filter is not None:
        u = u_filter(u)
    target = cen + r * u
    aim = _unit(u + 0.4 * _perp(rng, u))
    return target, aim * (0.2 if inside else 4.0), tm


def _aim_box(rng, lo, hi, xf, n, where):
    """Targets on a box in object space: 'face' interiors, 'edge' lines or 'corner' points; aim = the outward normals summed."""
    p = lo + rng.uniform(0.05, 0.95, (n, 3)) * (hi - lo)
    out = np.zeros((n, 3))
    k = {"face": 1, "edge": 2, "corner": 3}[where]
    for i in range(n):
        for ax in rng.permutation(3)[:k]:
            side = rng.integers(2)
            p[i, ax] = hi[ax] if side else lo[ax]
            out[i, ax] = 1.0 if side else -1.0
    aim = _unit(_unit(out) + 0.3 * _unit(rng.normal(size=(n, 3))))
    return xf.point(p), xf.point(aim, vec=True) * 4.0


def start_points(orc, n_per=1500, seed=11):
    """Adversarial start points: oracle hit points p = o + t d (ray::at) of rays aimed at each feature, with the primitive
    the oracle reports as the start primitive.  Returns the scene and a dict of arrays (p, start, time, target, type)."""
    s, desc, F = adversarial_scene()
    rng = np.random.default_rng(seed)
    T, A, TM, TY, IDS = [], [], [], [], []

    def add(kind, target, aim, tm, ids):
        T.append(target), A.append(aim), TM.append(tm), TY.extend([kind] * len(target))
        IDS.extend([tuple(ids)] * len(target))

    for kind, c, r, dc, pid in F["spheres"]:
        if kind == "ground":
            xz = rng.uniform(-8, 8, (n_per, 2))
            u = _unit(np.stack([xz[:, 0], np.full(n_per, 1000.0), xz[:, 1]], axis=1))
            target, tm = c + r * u, rng.uniform(0, 1, n_per)
            add("ground", target, _unit(u + 0.5 * _perp(rng, u)) * 4.0, tm, [pid])
            # touching: the ground right around the contact points of the resting spheres
            sm = [x for x in F["spheres"] if x[0] == "small"]
            k = rng.integers(len(sm), size=n_per)
            rho, phi = rng.uniform(0.002, 0.05, n_per), rng.uniform(0, 2 * np.pi, n_per)
            foot = np.array([sm[i][1] for i in k]) + np.stack([rho * np.cos(phi), np.zeros(n_per), rho * np.sin(phi)], 1)
            u = _unit(foot - c)
            target = c + r * u
            add("touching", target, _unit(u + 0.6 * _perp(rng, u)) * 0.3, rng.uniform(0, 1, n_per), [pid])
            continue
        m = max(n_per // sum(1 for x in F["spheres"] if x[0] == kind), 1)
        if kind == "small":
            target, aim, tm = _aim_sphere(rng, c, r, dc, m, lambda u: u * np.where(u[:, 1:2] < -0.3, -1.0, 1.0))
            add("small_sphere", target, aim, tm, [pid])
            def lower(u):  # 25-60 degrees off the contact point at the bottom
                th, ph = rng.uniform(0.44, 1.05, len(u)), rng.uniform(0, 2 * np.pi, len(u))
                return np.stack([np.sin(th) * np.cos(ph), -np.cos(th), np.sin(th) * np.sin(ph)], 1)
            target, aim, tm = _aim_sphere(rng, c, r, dc, m // 2, lower)
            add("touching", target, _unit(aim) * 0.04, tm, [pid])
        elif kind == "moving":
            add("moving_sphere", *_aim_sphere(rng, c, r, dc, m), [pid])
        elif kind == "nested_outer":
            add("nested_glass", *_aim_sphere(rng, c, r, dc, n_per // 2), [pid])
        else:
            add("nested_glass", *_aim_sphere(rng, c, r, dc, n_per // 2, inside=True), [pid])
    for kind, q, u, v, ids in F["quads"]:
        m = n_per // (8 if kind == "quad" else 1)
        nq = _unit(np.cross(u, v))
        for where in ("interior", "edge"):
            ab = rng.uniform(0.05, 0.95, (m, 2))
            if where == "edge":
                ab[np.arange(m), rng.integers(2, size=m)] = rng.integers(2, size=m).astype(np.float64)
            target = q + ab[:, :1] * u + ab[:, 1:] * v
            side = np.where(rng.random(m) < 0.5, -1.0, 1.0)[:, None]
            aim = _unit(side * nq + 0.5 * _perp(rng, np.broadcast_to(nq, (m, 3)).copy())) * 4.0
            add(kind if where == "interior" else "quad_edge", target, aim, rng.uniform(0, 1, m), ids)
    for _, lo, hi, xf, ids in F["boxes"]:
        for where in ("face", "edge", "corner"):
            target, aim = _aim_box(rng, lo, hi, xf, n_per // 3, where)
            add("box_" + where, target, aim, rng.uniform(0, 1, len(target)), ids)
    # touching: the top of the lower stacked box around the upper one's footprint, the upper one's sides near the seam
    (alo, ahi, xf, aids), (blo, bhi, _, bids) = F["stack"]
    m = n_per // 2
    ring = rng.uniform(0.0005, 0.05, m)
    side = rng.integers(4, size=m)
    t = rng.uniform(-0.5, 0.5, m)
    px = np.where(side == 0, 0.5 + ring, np.where(side == 1, -0.5 - ring, t))
    pz = np.where(side == 2, 0.5 + ring, np.where(side == 3, -0.5 - ring, t))
    target = xf.point(np.stack([px, np.ones(m), pz], 1))
    aim = xf.point(_unit(np.stack([np.zeros(m), np.ones(m), np.zeros(m)], 1) + 0.5 * _unit(rng.normal(size=(m, 3)))), vec=True) * 0.3
    add("touching", target, aim, rng.uniform(0, 1, m), aids)
    y = 1.0 + rng.uniform(0.0005, 0.05, m)
    nrm = np.zeros((m, 3))
    nrm[np.arange(m), np.where(side < 2, 0, 2)] = np.where(side % 2 == 0, 1.0, -1.0)
    p = np.stack([np.where(side == 0, 0.5, np.where(side == 1, -0.5, t)), y, np.where(side == 2, 0.5, np.where(side == 3, -0.5, t))], 1)
    add("touching", xf.point(p), xf.point(_unit(nrm + 0.5 * _unit(rng.normal(size=(m, 3)))), vec=True) * 0.3, rng.uniform(0, 1, m), bids)

    target, aim, tm = np.concatenate(T), np.concatenate(A), np.concatenate(TM)
    o = target + aim
    d = (target - o) * rng.uniform(0.3, 3.0, (len(o), 1))
    ids, t, nrm, _, _ = orc.hit_rays(desc, o, d, tm, 0.001, np.inf)
    p = o + t[:, None] * d  # ray::at
    ty = np.array(TY)
    on_feature = np.array([ids[i] in IDS[i] for i in range(len(ids))])
    keep = on_feature & (np.abs(p - target).max(axis=1) <= 1e-9 * SCALE)
    return s, desc, dict(p=p[keep], start=ids[keep], time=tm[keep], normal=nrm[keep], target=target[keep], type=ty[keep],
                         aimed=ty, landed=keep)


def bounce_rays(pts, seed=3):
    """Three directions per start point: outward, inward (log-uniform elevations >= 1e-3 rad off the tangent plane) and
    within 1e-3 rad of tangent, un-normalised.  Returns (origin, direction, time, start id, type, direction class)."""
    rng = np.random.default_rng(seed)
    n = len(pts["p"])
    nrm = _unit(pts["normal"])
    cols = []
    for cls in DIR_CLASSES:
        if cls == "tangent":
            e = rng.uniform(-1e-3, 1e-3, n)
        else:
            e = np.exp(rng.uniform(np.log(1e-3), np.log(np.pi / 2), n)) * (1.0 if cls == "out" else -1.0)
        d = np.cos(e)[:, None] * _perp(rng, nrm) + np.sin(e)[:, None] * nrm
        cols.append((d * rng.uniform(0.3, 3.0, (n, 1)), np.full(n, cls)))
    d = np.concatenate([c[0] for c in cols])
    rep = lambda a: np.concatenate([a] * len(DIR_CLASSES))  # noqa: E731
    return rep(pts["p"]), d, rep(pts["time"]), rep(pts["start"]), rep(pts["type"]), np.concatenate([c[1] for c in cols])


def leaf_rule_table(rtb, orc, ctx, n_per=1500):
    """Per (start type, direction class): rays, id agreement, self disagreements, t p99.9 (relative, agreeing hits)."""
    s, desc, pts = start_points(orc, n_per)
    ctx.upload_scene(desc)
    o, d, tm, start, ty, cls = bounce_rays(pts)
    ids, t, _, _ = ctx.trace_rays(o, d, tm, 0.001, np.inf, rtb.RT_TRACE_FP32, start_prim=start)
    oi, ot, *_ = orc.hit_rays(desc, o, d, tm, 0.001, np.inf)
    table = {}
    for key in sorted(set(zip(ty, cls))):
        m = (ty == key[0]) & (cls == key[1])
        agree = ids[m] == oi[m]
        self_dis = int(((ids[m] == start[m]) != (oi[m] == start[m])).sum())
        ok = agree & (oi[m] >= 0)
        rel = np.abs(t[m][ok] - ot[m][ok]) / np.abs(ot[m][ok])
        table[key] = dict(n=int(m.sum()), agree=float(agree.mean()), self=self_dis, t_p999=float(np.quantile(rel, 0.999)) if ok.any() else 0.0)
    return table


# ---- (a) the leaf rules on adversarial start points ------------------------------------------------------------
# Measured on a B200 (profiles/r3_bounce_parity.md); the bounds are the measurement + 25 %.  Self disagreements: 0 in every
# class, edges, corners and tangents included, so every class is held at 0.  Id agreement is >= 0.999 except where a
# start point touches another primitive: a coincident quad pair and boxes stacked face to face meet at exactly equal t
# (the reference breaks that tie by list order, fp32 by rounding), and the fp32 rounding of a start point on one of two
# coincident quads puts the twin 1e-3 ahead of a near-tangent ray.  Those classes are held to their measured mismatch
# counts.  t p99.9 is <= 1e-4 except where the answer itself is ill-conditioned in the start point: a chord of a small
# sphere or a hit at grazing incidence moves by |fp32 rounding of p| / sin(elevation)^k, and the kernel traces the fp32 p.
MISMATCH_MAX = {
    ('quad_coincident', 'out'): 3,
    ('quad_coincident', 'tangent'): 155,
    ('quad_edge', 'tangent'): 53,
    ('touching', 'in'): 243,
    ('touching', 'tangent'): 125,
}
T_P999_MAX = {
    ('ground', 'tangent'): 0.001,
    ('moving_sphere', 'in'): 0.0013,
    ('moving_sphere', 'tangent'): 0.0025,
    ('nested_glass', 'in'): 0.0012,
    ('nested_glass', 'tangent'): 0.00066,
    ('quad', 'in'): 0.0042,
    ('quad', 'out'): 0.0013,
    ('quad', 'tangent'): 0.0017,
    ('quad_edge', 'in'): 0.00029,
    ('small_sphere', 'in'): 0.0021,
    ('small_sphere', 'out'): 0.0018,
    ('small_sphere', 'tangent'): 0.0026,
    ('touching', 'in'): 0.003,
    ('touching', 'out'): 0.0038,
    ('touching', 'tangent'): 0.0028,
}


def test_adversarial_start_points_lie_on_their_features(orc):
    """CPU: every kept start point is the oracle's hit on the feature it was aimed at (within 1e-9 of the aimed point), and
    enough of every feature's aimed rays land there for the per-class gates to mean something."""
    s, desc, pts = start_points(orc)
    aimed, landed = pts["aimed"], pts["landed"]
    for kind in sorted(set(aimed)):
        frac = landed[aimed == kind].mean()
        assert frac >= 0.3, (kind, frac)
        assert (pts["type"] == kind).sum() >= 300, kind
    # the oracle's own check of an interior start point: a short ray back into the surface from 1e-3 above it hits the
    # start primitive at t = 1 (at an edge or corner it may as well hit the neighbouring face or slip past)
    interior = ~np.isin(pts["type"], EDGE_TYPES)
    assert interior.sum() > 0 and (~interior).sum() > 0
    n = _unit(pts["normal"][interior])
    ids, t, *_ = orc.hit_rays(desc, pts["p"][interior] + 1e-3 * n, -1e-3 * n, pts["time"][interior], 1e-6, np.inf)
    assert np.array_equal(ids, pts["start"][interior])
    assert np.abs(t - 1.0).max() <= 1e-6


@pytest.mark.gpu
def test_start_primitive_rules_match_the_oracle(rtb, orc, gpu_ctx):
    table = leaf_rule_table(rtb, orc, gpu_ctx)
    assert len(table) == 11 * len(DIR_CLASSES)
    for (ty, cls), r in table.items():
        assert r["self"] == 0, (ty, cls, r)
        assert r["agree"] >= 0.999 or round((1 - r["agree"]) * r["n"]) <= MISMATCH_MAX.get((ty, cls), -1), (ty, cls, r)
        assert r["t_p999"] <= T_P999_MAX.get((ty, cls), 1e-4), (ty, cls, r)


@pytest.mark.gpu
def test_start_prim_arguments(rtb, orc, gpu_ctx):
    s, desc, F = adversarial_scene()
    gpu_ctx.upload_scene(desc)
    o, d = np.zeros((2, 3)), np.ones((2, 3))
    with pytest.raises(rtb.RtError):  # the exact path is the reference: no start primitive there
        gpu_ctx.trace_rays(o, d, None, 0.001, np.inf, rtb.RT_TRACE_EXACT, start_prim=[-1, -1])
    with pytest.raises(rtb.RtError):
        gpu_ctx.trace_rays(o, d, start_prim=[-1, s.n_prims])
    with pytest.raises(rtb.RtError):
        gpu_ctx.trace_rays(o, d, start_prim=[-1, -7])
    a = gpu_ctx.trace_rays(o, d, start_prim=[-1, -1])
    b = gpu_ctx.trace_rays(o, d)
    assert all(np.array_equal(x, y) for x, y in zip(a, b))


# ---- (b) the render kernel's own bounce rays ---------------------------------------------------------------------
def center_rays(orc, cam):
    """Pixel-centre rays in numpy with center_rays_kernel's operation order (camera.hpp:147,156), H*W x 3 each."""
    f = orc.camera_frame(cam)
    h, w = orc.image_height(cam), cam.image_width
    v = lambda a: np.array(a[:], np.float64)  # noqa: E731
    j, i = np.meshgrid(np.arange(h, dtype=np.float64), np.arange(w, dtype=np.float64), indexing="ij")
    ps = v(f.pixel00_loc) + (i.reshape(-1, 1) + 0.0) * v(f.pixel_delta_u) + (j.reshape(-1, 1) + 0.0) * v(f.pixel_delta_v)
    c = np.broadcast_to(v(f.center), ps.shape).copy()
    return c, ps - c


def material_kinds(rtb, desc):
    """prim id -> rt_material.kind of the scene description."""
    d = desc.contents
    kinds = {}
    for k in range(d.n_hittables):
        h = d.hittables[k]
        if h.prim_id >= 0 and h.material >= 0:
            kinds[h.prim_id] = d.materials[h.material].kind
    return kinds


def bounce_parity(rtb, orc, ctx, desc, cam, seed=1):
    """The kernel's bounce segment against orc.hit_rays from the oracle's primary hit point along the kernel's d1."""
    ctx.upload_scene(desc)
    out = ctx.bounce_visibility(cam, seed)
    c, dirs = center_rays(orc, cam)
    oid, ot, *_ = orc.hit_rays(desc, c, dirs, None, 0.001, np.inf, skip_media=True)
    gid = out["id"].reshape(-1)
    id1, t1 = out["id1"].reshape(-1), out["t1"].reshape(-1)
    o1, d1 = out["o1"].reshape(-1, 3).astype(np.float64), out["d1"].reshape(-1, 3).astype(np.float64)
    hit = (gid == oid) & (oid >= 0)
    kinds = material_kinds(rtb, desc)
    kind = np.array([kinds.get(int(x), 0) for x in oid])
    nob = id1 == rtb.RT_NO_BOUNCE
    absorbing = np.isin(kind, (rtb.RT_M_DIFFUSE_LIGHT, rtb.RT_M_METAL))
    m = hit & ~nob
    p64 = c[m] + ot[m][:, None] * dirs[m]  # ray::at
    rid, rt_, _, rff, _ = orc.hit_rays(desc, p64, d1[m], None, 0.001, np.inf, skip_media=True)
    start, gi, gt, gff = oid[m], id1[m], t1[m], out["front1"].reshape(-1)[m]
    agree = gi == rid
    ok = agree & (rid >= 0)
    rel = np.abs(gt[ok] - rt_[ok]) / np.abs(rt_[ok])
    dp = np.abs(o1[m] - p64).max(axis=1) / np.maximum(1.0, np.abs(p64).max(axis=1))
    q = lambda a, x: float(np.quantile(a, x)) if a.size else 0.0  # noqa: E731
    return dict(pixels=int(gid.size), primary_skipped=int((gid != oid).sum()), bounces=int(m.sum()), id_mismatch=int((~agree).sum()),
                self=int(((gi == start) != (rid == start)).sum()), t_p999=q(rel, 0.999), t_max=float(rel.max()) if rel.size else 0.0,
                front_mismatch=int((gff[ok] != rff[ok]).sum()), p_p999=q(dp, 0.999), p_max=float(dp.max()) if dp.size else 0.0,
                no_bounce=int((hit & nob).sum()), no_bounce_wrong=int((hit & nob & ~absorbing).sum() + (hit & ~nob & (kind == rtb.RT_M_DIFFUSE_LIGHT)).sum()),
                miss_no_bounce=bool(np.all(nob[oid < 0] | (gid[oid < 0] >= 0))))


def constructed_scenes():
    """(name, desc, camera) of the three scenes built for the bounce gate."""
    out = []
    s = su.SceneDesc()
    floor, white = s.lambertian(s.solid(0.4, 0.5, 0.3)), s.lambertian(s.solid(0.7, 0.7, 0.7))
    glass = s.dielectric(1.5)
    kids = [s.quad((-20, 0, -20), (40, 0, 0), (0, 0, 40), floor), s.quad((-2, 6, -2), (4, 0, 0), (0, 0, 4), s.light(s.solid(4, 4, 4)))]
    kids.append(s.translate(s.rotate_y(s.box((-1, 0, -1), (1, 2, 1), glass), 23.0), (-1.5, 0, 0)))
    kids.append(s.translate(s.box((0, 0, 0), (1.5, 1, 1.5), white), (1.5, 0, -1)))
    kids.append(s.translate(s.rotate_y(s.box((0, 0, 0), (1, 1, 1), white), -17.0), (1.75, 1, -0.75)))
    out.append(("dielectric_boxes", s, s.finish(s.list(kids)), su.camera(width=480, aspect=1.5, depth=8, lookfrom=(3, 4, 9), lookat=(0, 0.8, 0), vfov=35.0)))
    s = su.SceneDesc()
    ground, glass, red = s.lambertian(s.checker(0.5, s.solid(0.2, 0.3, 0.1), s.solid(0.9, 0.9, 0.9))), s.dielectric(1.5), s.lambertian(s.solid(0.7, 0.2, 0.2))
    kids = [s.sphere((0, -1000, 0), 1000, ground), s.sphere((-2.5, 1.2, 0), 1.2, glass), s.sphere((-2.5, 1.2, 0), 0.8, glass), s.sphere((-2.5, 1.2, 0), -0.6, glass),
            s.sphere((2, 2, 0), 2.0, red)]
    rng = np.random.default_rng(4)
    for th, ph in zip(rng.uniform(0, 0.9, 24), rng.uniform(0, 2 * np.pi, 24)):
        u = np.array([np.sin(th) * np.cos(ph), np.cos(th), np.sin(th) * np.sin(ph)])
        kids.append(s.sphere(tuple(np.array([2, 2, 0]) + 2.1 * u), 0.1, glass if th < 0.3 else red))
    out.append(("nested_glass", s, s.finish(s.list(kids)), su.camera(width=480, aspect=1.5, depth=8, lookfrom=(0, 3, 10), lookat=(0, 1.5, 0), vfov=40.0)))
    s = su.SceneDesc()
    metal, polished = s.metal((0.8, 0.8, 0.9), 0.4), s.metal((0.9, 0.7, 0.5), 0.05)
    kids = [s.quad((-50, 0, -50), (100, 0, 0), (0, 0, 100), metal), s.quad((-3, 0.01, -30), (0, 3, 0), (6, 0, 0), s.light(s.solid(3, 3, 3)))]
    for k in range(10):
        kids.append(s.sphere((float(k % 5) * 2.0 - 4.0, 0.5, -3.0 * (k // 5) - 2.0), 0.5, metal if k % 2 else polished))
    out.append(("grazing_metal", s, s.finish(s.list(kids)), su.camera(width=480, aspect=2.0, depth=8, lookfrom=(0, 0.25, 6), lookat=(0, 0.2, -10), vfov=30.0)))
    return out


# scene -> metric -> bound: the B200 measurement + 25 % (tools/bounce_parity.py, profiles/r3_bounce_parity.md).  Id mismatches:
# dielectric_boxes 2494 — rays refracted into the glass box reach its bottom face, which lies on the floor quad (an exact tie
# the reference gives to the later primitive; not verified pixel by pixel) —, book1_final 15, nested_glass 1, none elsewhere.
BOUNCE_MAX = {
    'bouncing_spheres': {'id_mismatch': 0, 't_p999': 0.0078, 't_max': 0.03, 'front_mismatch': 0, 'p_p999': 7.6e-05, 'p_max': 0.0001},
    'checkered_spheres': {'id_mismatch': 0, 't_p999': 1.1e-05, 't_max': 5.1e-05, 'front_mismatch': 0, 'p_p999': 3.5e-06, 'p_max': 6.2e-05},
    'earth': {'id_mismatch': 0, 't_p999': 1.2e-07, 't_max': 1.2e-07, 'front_mismatch': 0, 'p_p999': 3.5e-06, 'p_max': 2.3e-05},
    'perlin_sphere': {'id_mismatch': 0, 't_p999': 0.0026, 't_max': 0.0036, 'front_mismatch': 0, 'p_p999': 0.00012, 'p_max': 0.00013},
    'quads': {'id_mismatch': 0, 't_p999': 8.3e-07, 't_max': 9.3e-07, 'front_mismatch': 0, 'p_p999': 4.5e-07, 'p_max': 4.5e-07},
    'simple_light': {'id_mismatch': 0, 't_p999': 0.0025, 't_max': 0.0029, 'front_mismatch': 0, 'p_p999': 0.00011, 'p_max': 0.00013},
    'cornell_box': {'id_mismatch': 0, 't_p999': 0.02, 't_max': 0.022, 'front_mismatch': 0, 'p_p999': 2.6e-06, 'p_max': 2e-05},
    'book1_final': {'id_mismatch': 19, 't_p999': 0.0079, 't_max': 0.086, 'front_mismatch': 0, 'p_p999': 0.0001, 'p_max': 0.0024},
    'cornell_rotated': {'id_mismatch': 0, 't_p999': 0.02, 't_max': 0.022, 'front_mismatch': 0, 'p_p999': 2.6e-06, 'p_max': 2e-05},
    'cornell_smoke': {'id_mismatch': 0, 't_p999': 0.02, 't_max': 0.022, 'front_mismatch': 0, 'p_p999': 2.6e-06, 'p_max': 2e-05},
    'book2_final': {'id_mismatch': 0, 't_p999': 0.0003, 't_max': 0.12, 'front_mismatch': 0, 'p_p999': 2.4e-06, 'p_max': 9.4e-06},
    'dielectric_boxes': {'id_mismatch': 3118, 't_p999': 0.00025, 't_max': 0.0048, 'front_mismatch': 0, 'p_p999': 1.3e-06, 'p_max': 2e-06},
    'nested_glass': {'id_mismatch': 2, 't_p999': 0.0024, 't_max': 0.0051, 'front_mismatch': 0, 'p_p999': 0.00012, 'p_max': 0.00013},
    'grazing_metal': {'id_mismatch': 0, 't_p999': 2.8e-05, 't_max': 8.4e-05, 'front_mismatch': 0, 'p_p999': 2.1e-06, 'p_max': 3.9e-06},
}


def _check_bounce(name, r):
    bound = BOUNCE_MAX[name]
    assert r["miss_no_bounce"] and r["no_bounce_wrong"] == 0, (name, r)
    assert r["self"] == 0, (name, r)
    assert r["bounces"] > 0.2 * (r["pixels"] - r["primary_skipped"]) or name in ("earth", "simple_light"), (name, r)
    for key in ("id_mismatch", "t_p999", "t_max", "front_mismatch", "p_p999", "p_max"):
        assert r[key] <= bound[key], (name, key, r[key], bound[key])


@pytest.mark.gpu
@pytest.mark.parametrize("name", ALL_SCENES)
def test_render_kernel_bounce_matches_oracle(rtb, orc, gpu_ctx, name):
    sc = rtb.Scene(name, rand_seed=1)
    _check_bounce(name, bounce_parity(rtb, orc, gpu_ctx, sc.desc, sc.camera_copy()))


@pytest.mark.gpu
@pytest.mark.parametrize("which", range(3))
def test_render_kernel_bounce_on_constructed_scenes(rtb, orc, gpu_ctx, which):
    name, s, desc, cam = constructed_scenes()[which]
    _check_bounce(name, bounce_parity(rtb, orc, gpu_ctx, desc, cam))


def test_center_rays_reproduce_oracle_primary(rtb, orc):
    """CPU: the numpy pixel-centre rays fed to orc.hit_rays are orc.primary bit for bit (so part (b)'s p64 is the oracle's
    own primary hit point)."""
    for name, width in (("cornell_box", 120), ("book1_final", 160), ("book2_final", 100), ("quads", 90)):
        sc = rtb.Scene(name, rand_seed=1)
        cam = sc.camera_copy(image_width=width)
        c, d = center_rays(orc, cam)
        ids, t, nrm, _, _ = orc.hit_rays(sc.desc, c, d, None, 0.001, np.inf, skip_media=True)
        pid, pt, pn = orc.primary(sc.desc, cam, skip_media=True)
        assert np.array_equal(ids, pid.reshape(-1)) and (pid >= 0).any(), name
        assert np.array_equal(t, pt.reshape(-1)) and np.array_equal(nrm, pn.reshape(-1, 3)), name
    for name, s, desc, cam in constructed_scenes():
        c, d = center_rays(orc, cam)
        ids, *_ = orc.hit_rays(desc, c, d, None, 0.001, np.inf, skip_media=True)
        assert np.array_equal(ids, orc.primary(desc, cam)[0].reshape(-1)) and (ids >= 0).mean() > 0.5, name


# ---- (c) one scene, every plan ------------------------------------------------------------------------------------
@contextlib.contextmanager
def knob_context(rtb, knob):
    """A fresh Context created with the environment knob `knob` set (rt_init reads the knobs once)."""
    old = os.environ.get(knob) if knob else None
    if knob:
        os.environ[knob] = "1"
    try:
        ctx = rtb.Context(0)
    finally:
        if knob:
            if old is None:
                del os.environ[knob]
            else:
                os.environ[knob] = old
    try:
        yield ctx
    finally:
        ctx.close()


PLAN_SCENES = ["bouncing_spheres", "book1_final", "book2_final", "perlin_sphere", "cornell_smoke"]
PLAN_KNOBS = [None, "RT_B200_NO_STAGING", "RT_B200_NO_SMEM_STACK"]


def plan_outputs(rtb, name, width=160, spp=16, seed=3):
    sc = rtb.Scene(name, rand_seed=1)
    cam = sc.camera_copy(image_width=width, samples_per_pixel=spp)
    res = {}
    for knob in PLAN_KNOBS:
        with knob_context(rtb, knob) as ctx:
            ctx.upload_scene(sc.desc)
            ctx.render(cam, seed=seed, flags=rtb.RT_RENDER_MEGAKERNEL)
            res[knob or "default"] = dict(accum=ctx.download_accum(), rays=ctx.stats().rays, aov=ctx.bounce_visibility(cam, seed))
            if knob is None:
                ctx.render(cam, seed=seed, flags=rtb.RT_RENDER_MEGAKERNEL | rtb.RT_RENDER_COUNTERS)
                st = ctx.stats()
                res["counters"] = dict(accum=ctx.download_accum(), rays=st.rays, census=np.array(st.census[:], np.int64))
    return res


@pytest.mark.gpu
@pytest.mark.parametrize("name", PLAN_SCENES)
def test_every_plan_renders_the_same_bits(rtb, name):
    """The plans move nodes and stacks, not the primitive a ray ends on: accumulators, ray counts and the bounce AOV are
    bit-identical under every megakernel plan and the instrumented kernel."""
    res = plan_outputs(rtb, name)
    ref = res["default"]
    assert ref["accum"].any() and ref["rays"] > 0
    for plan, r in res.items():
        assert np.array_equal(r["accum"], ref["accum"]), (name, plan, int((r["accum"] != ref["accum"]).sum()))
        assert r["rays"] == ref["rays"], (name, plan)
        if "aov" in r:
            for key, a in r["aov"].items():
                assert np.array_equal(a, ref["aov"][key]), (name, plan, key)
    cn, rays = res["counters"]["census"], res["counters"]["rays"]
    assert cn[0] > 0, cn  # node visits
    assert cn[2] <= cn[1] and cn[4] <= cn[3], cn  # sphere hits <= tests, full quad tests <= quad tests
    assert cn[6:11].sum() <= rays and cn[6:11].sum() > 0, (cn, rays)  # every scatter follows a ray
