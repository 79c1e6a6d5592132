"""Boundary rays: pairs of rays, adjacent floats apart, on the two sides of a decision of the reference's World::hit —
sphere tangency, root choice, the sphere and mesh windows, the triangle's parallel and edge tests, the CULL bound and
the tiny-origin fallback — and rays whose hits are exact ties between primitives.

Every exact walk puts a shortcut in front of the reference's own arithmetic (the FILTER walk's FFMA2 discriminant
bound, the CULL walk's group bound, the triangle plane stage's widened window and edge stage's half-height margin,
the any-hit exit, the out-of-order sphere visits of the CULL walk and of the DIRECT group's second pass).  Each is
correct because of a margin or a tie rule; these rays sit where a weakened margin or a dropped tie rule changes the
answer, where the seeded families of test_rays.py only come close.

The generator is CPU-only, seeded and deterministic.  A family is a ray in which one float (an origin, t_max or
direction component) varies between two values whose reference records differ (another prim, or a depth more than a
few ulps away: a root choice).  Bisection over the float's bit pattern, one batched `rays_reference` call per step
for all the families of a world, ends on two adjacent floats; both rays are kept.  Coverage is asserted, not hoped
for: every pair straddles its decision under the reference and under test_rays.literal_hit, each regime yields a
stated number of pairs, and the tangency pairs sit within 64u(o.o + c.c + r^2) of the exact discriminant on both
sides (u = 2^-24), inside the filter's 128u margin.

CPU tests: ray_hit and ray_occluded of rt_trace.cuh built for the host (tests/rays_host, tests/occlusion_host), plain
and with the reciprocal approximation moved +-1 ulp, for the DIRECT, FILTER and CULL walks; tie worlds rendered by
tests/hostsim at fixed jitter for every walk.  GPU tests: the ray and occlusion kernels on every set (DIRECT below 64
spheres, FILTER and CULL with the lists staged in shared memory and read from global memory) and the exact render of
the tie worlds through each walk row.
"""
import ctypes as C
import os
import subprocess
import sys
from fractions import Fraction
from pathlib import Path

import numpy as np
import pytest

import test_occlusion
import test_rays
from test_rays import F, INF, NAMES, _rays, assert_same, literal_records, reference

HERE = Path(__file__).resolve().parent
ROOT = HERE.parent
U = Fraction(1, 2 ** 24)
DIRECT, FILTER, CULL, NP2 = 0, 0x80000000, 0x40000000, 0x20000000
FILTER_FROM = 64
GLOBAL_SPHERES = 16000           # hot lists of the FILTER and CULL walks larger than a B200's shared memory
MATERIALS = ("material M0 : Diffuse color 0.7 0.3 0.2;\nmaterial M1 : Metal color 0.8 0.8 0.9 fuzz 0.2;\n"
             "material M2 : Dielectric ir 1.5;\nmaterial M3 : Diffuse color 0.1 0.6 0.3;\n"
             "material M4 : Metal color 0.9 0.5 0.1 fuzz 0.0;\n")


# ------------------------------------------------------------------------------------------------ float bit patterns

def keys(x):
    """Monotone integer keys of float32 values: adjacent floats have adjacent keys (+0 and -0 share 0)."""
    b = np.asarray(x, np.float32).view(np.uint32).astype(np.int64)
    return np.where(b < 2 ** 31, b, -(b & 0x7FFFFFFF))


def floats(k):
    k = np.asarray(k, np.int64)
    return np.where(k >= 0, k, 0x80000000 | -k).astype(np.uint32).view(np.float32)


def fmt(x):
    """A float32 in the world grammar's positional form (no exponent), with enough digits to read back the same bits."""
    return np.format_float_positional(F(x), unique=True, trim="0")


# ---------------------------------------------------------------------------------------------------------- worlds

class World:
    """A world built from float32 values: its text, and the bits the text must read back as."""

    def __init__(self, camera=(0.0, 0.0, 0.0)):
        self.camera = tuple(F(c) for c in camera)
        self.spheres, self.triangles = [], []

    def sphere(self, c, r, m=0):
        self.spheres.append((tuple(F(x) for x in c), F(r), m))
        return len(self.spheres) - 1

    def triangle(self, v0, v1, v2, m=1):
        self.triangles.append(tuple(tuple(F(x) for x in v) for v in (v0, v1, v2)) + (m,))
        return len(self.triangles) - 1

    def text(self, fill=0):
        lines = [f"camera origin {' '.join(map(fmt, self.camera))} aspect 1.5;", MATERIALS]
        for c, r, m in self.spheres + self.fillers(fill):
            lines.append(f"sphere center {' '.join(map(fmt, c))} radius {fmt(r)} material M{m};")
        for v0, v1, v2, m in self.triangles:
            lines.append("triangle " + " ".join(f"v{k} {' '.join(map(fmt, v))}" for k, v in enumerate((v0, v1, v2)))
                         + f" material M{m};")
        return "\n".join(lines) + "\n"

    def fillers(self, n):
        """n spheres of the median radius far outside the world (they change the walk, not the answers near it):
        the CULL walk's groups keep members of the world's own size."""
        if n <= 0:
            return []
        rng = np.random.default_rng(977)
        radii = np.abs([r for _, r, _ in self.spheres] or [F(1)])
        r = F(np.median(radii))
        pts = [c for c, _, _ in self.spheres] + [v for t in self.triangles for v in t[:3]]
        ext = max([float(np.max(np.abs(p))) for p in pts] + [1.0])
        v = rng.normal(size=(n, 3))
        c = (v / np.linalg.norm(v, axis=1, keepdims=True) * (1e3 * ext + 1e3 * float(r))).astype(np.float32)
        return [(tuple(ci), r, 4) for ci in c]

    def n_fill_wide(self):
        return max(0, FILTER_FROM + 8 - len(self.spheres))

    def n_fill_global(self):
        return GLOBAL_SPHERES - len(self.spheres)


def parse_exact(ob, w, fill=0):
    """The oracle's world of w.text(fill), asserting that it holds the intended float32 bits."""
    text = w.text(fill)
    cam, world = ob.parse_input(text)
    want_s = w.spheres + w.fillers(fill)
    got_s = world.spheres()
    assert len(got_s) == len(want_s) and world.n_triangles == len(w.triangles)
    for s, (c, r, _) in zip(got_s, want_s):
        assert np.array_equal(np.array(s.center.tuple() + (s.radius,), np.float32).view(np.uint32),
                              np.array(c + (r,), np.float32).view(np.uint32)), (s.center.tuple(), s.radius, c, r)
    for t, (v0, v1, v2, _) in zip(world.triangles(), w.triangles):
        got = np.array(t.v0.tuple() + t.v1.tuple() + t.v2.tuple(), np.float32).view(np.uint32)
        assert np.array_equal(got, np.array(v0 + v1 + v2, np.float32).view(np.uint32))
    return text, cam, world


# -------------------------------------------------------------------------------------------------------- bisection

def _ray(o, a, t_max=INF):
    r = np.zeros(8, np.float32)
    r[0:3], r[3], r[4:7] = o, t_max, a
    return r


def _differ(a, b, i=slice(None), j=slice(None)):
    """Records that differ: another prim, or a depth more than 4 ulps away (the other root)."""
    return (a["prim"][i] != b["prim"][j]) | (np.abs(keys(a["depth"][i]) - keys(b["depth"][j])) > 4)


def _put(rec, mask, src):
    for k in NAMES:
        rec[k][mask] = src[k][mask]


def bisect(ob, world, fams):
    """fams: [(ray, component, value_a, value_b, tag)].  Returns (pairs [m, 2, 8], tags) of the families whose end
    records differ, each pair two rays that are adjacent floats in the family's component with differing records."""
    if not fams:
        return np.zeros((0, 2, 8), np.float32), []
    base = np.array([f[0] for f in fams], np.float32)
    comp = np.array([f[1] for f in fams])
    ka, kb = keys([f[2] for f in fams]), keys([f[3] for f in fams])
    idx = np.arange(len(fams))

    def rays_at(k):
        r = base.copy()
        r[idx, comp] = floats(k)
        return r

    ra, rb = reference(ob, world, rays_at(ka)), reference(ob, world, rays_at(kb))
    alive = _differ(ra, rb)
    for _ in range(80):
        active = alive & (np.abs(ka - kb) > 1)
        if not active.any():
            break
        km = ka + (kb - ka) // 2
        rm = reference(ob, world, rays_at(km))
        # a change of prim is the decision when there is one; with one prim throughout, a jump of the depth is
        pm, pa, pb = rm["prim"], ra["prim"], rb["prim"]
        da, db = _differ(rm, ra), _differ(rm, rb)
        to_a = active & ((pm != pb) | ((pm == pa) & db))
        to_b = active & ~to_a & ((pm != pa) | da)
        alive &= ~(active & ~to_a & ~to_b)         # within a few ulps of both ends: no clean crossing here
        ka, kb = np.where(to_a, km, ka), np.where(to_b, km, kb)
        _put(ra, to_a, rm)
        _put(rb, to_b, rm)
    alive &= np.abs(ka - kb) == 1
    pairs = np.stack([rays_at(ka), rays_at(kb)], axis=1)[alive]
    return pairs, [f[4] for f, a in zip(fams, alive) if a]


# --------------------------------------------------------------------------------------------------------- regimes
# Each returns (World, families, extra rays).  A family's tag names the sphere whose tangency it crosses (or None).

def _unit(rng):
    v = rng.normal(size=3)
    return v / np.linalg.norm(v)


def _tangency_families(rng, w, spheres, origins, fams, per=1):
    """Direction-varied and origin-varied crossings of the tangency of each listed sphere from each origin."""
    for i in spheres:
        c, r, _ = w.spheres[i]
        r = abs(float(r))
        for o in origins:
            o = np.asarray(o, np.float64)
            for _ in range(per):
                jitter = _unit(rng) * r * rng.uniform(0, 0.5)
                a = (np.asarray(c, np.float64) + jitter - o).astype(np.float32)
                k = int(np.argmin(np.abs(a)))
                sgn = rng.choice([-1.0, 1.0])
                for s in (1.5, 6.0, 40.0, 400.0):                     # the far side of the tangent
                    fams.append((_ray(o, a), 4 + k, a[k], F(float(a[k]) + sgn * s * r), i))
                if np.max(np.abs(o)) < 2.0 ** 30:
                    ko = int(np.argmin(np.abs(a)))
                    for s in (1.5, 6.0):
                        fams.append((_ray(o, a), ko, F(o[ko]), F(float(o[ko]) + sgn * s * r), i))


def regime_tangent_unit(rng, negative=False):
    w = World()
    for _ in range(6):
        c = (rng.uniform(-2, 2), rng.uniform(-1, 1), rng.uniform(-7, -3))
        r = rng.uniform(0.2, 1.0)
        w.sphere(c, -r if negative else r, int(rng.integers(0, 4)))
    fams = []
    origins = [rng.uniform(-0.5, 0.5, 3) for _ in range(3)]
    _tangency_families(rng, w, range(6), origins, fams)
    return w, fams, []


def regime_tangent_ground(rng):
    w = World()
    g = w.sphere((0.0, -1000.0, 0.0), 1000.0, 0)
    w.sphere((0.0, 1.0, -6.0), 0.5, 1)
    fams = []
    for h in (0.002, 0.01, 0.1, 1.0, 10.0):
        for _ in range(4):
            o = np.array([rng.uniform(-5, 5), h * rng.uniform(1, 2), rng.uniform(-5, 5)], np.float32)
            th = rng.uniform(0, 2 * np.pi)
            a = np.array([np.cos(th), -0.3, np.sin(th)], np.float32)
            fams.append((_ray(o, a), 5, F(-0.3), F(0.05), g))             # direction y from below to above the tangent
            s = rng.uniform(0.005, 0.05)
            a2 = np.array([np.cos(th), -s, np.sin(th)], np.float32)
            hstar = 1000.0 * (np.sqrt(1 + s * s) - 1.0)                    # the origin height of the tangent line
            fams.append((_ray(o, a2), 1, F(hstar * 0.25), F(hstar * 4.0), g))
    return w, fams, []


def regime_tangent_far(rng):
    w = World()
    radii = (1.0, 1000.0, 1.0e6, 2.0 ** 30)
    for k, r in enumerate(radii):
        w.sphere((0.0, 0.0, 0.0) if k == 0 else tuple(rng.uniform(-1, 1, 3) * r * 4), r, k % 4)
    fams = []
    for i, r in enumerate(radii):
        c = np.asarray(w.spheres[i][0], np.float64)
        for L in (2.0 ** 20, 2.0 ** 30, 2.0 ** 40):
            for j in range(3):
                o = c.copy()
                o[j] = rng.choice([-1.0, 1.0]) * L
                o[(j + 1) % 3] += rng.uniform(-0.5, 0.5) * r
                o = np.clip(o, -2.0 ** 40, 2.0 ** 40).astype(np.float32)
                a = (c - o).astype(np.float32)
                k = (j + 1 + int(rng.integers(0, 2))) % 3
                for s in (1.5, 6.0, 40.0):
                    fams.append((_ray(o, a), 4 + k, a[k], F(float(a[k]) + s * r), i))
    return w, fams, []


def regime_tangent_big_c(rng):
    w = World()
    for k in range(6):
        d = _unit(rng)
        d[2] = -abs(d[2])
        w.sphere(d * 10.0 ** rng.uniform(4, 6), 10.0 ** rng.uniform(-2, 0), k % 4)
    fams = []
    _tangency_families(rng, w, range(6), [rng.uniform(-0.5, 0.5, 3) for _ in range(2)], fams)
    return w, fams, []


def regime_root_choice(rng):
    """Origins on a sphere's surface: root1 crossing 0.001 (t jumps from root2 to root1) going in, root2 crossing
    0.001 (a hit or not) going out; plus rays from the surface point and a few ulps inside and outside it."""
    w = World()
    radii = (0.05, 1.0, 50.0, -2.0)
    for k, r in enumerate(radii):
        w.sphere((k * 200.0 - 300.0, rng.uniform(-1, 1), -20.0 - k * 100.0), r, k % 4)
    fams, extra = [], []
    for i, r in enumerate(radii):
        c = np.asarray(w.spheres[i][0], np.float64)
        for _ in range(6):
            nrm = _unit(rng)
            p = (c + abs(r) * nrm).astype(np.float32)
            for inward in (True, False):
                d = _unit(rng)
                if (d @ nrm < 0) != inward:
                    d = d - 2 * (d @ nrm) * nrm
                if abs(d @ nrm) < 0.2:
                    d = d - nrm * (0.4 if inward else -0.4)
                d = (d / np.linalg.norm(d)).astype(np.float32)
                k = int(np.argmax(np.abs(d)))
                # moving the origin by x e_k moves the near root by -x d_k
                if inward:
                    lo, hi = F(p[k] + 0.0005 / d[k]), F(p[k] - 0.004 / d[k])
                else:
                    lo, hi = F(p[k] - 0.004 / d[k]), F(p[k] + 0.0005 / d[k])
                fams.append((_ray(p, d), k, lo, hi, None))
                for m in (0, 1, 2, 4, -1, -2, -4):
                    q = p.copy()
                    q[k] = floats(keys(p[k]) + m)
                    extra.append(_ray(q, d))
    return w, fams, extra


def regime_sphere_window(rng):
    """Two spheres whose hits meet: side by side (the winner flips between adjacent t), in both list orders, and
    nested spheres touching at one point (an exact tie on the axis ray), in both list orders."""
    w = World()
    fams, extra = [], []
    for first in (0, 1):
        for _ in range(3):
            c = np.array([rng.uniform(-3, 3), rng.uniform(-2, 2), rng.uniform(-9, -5)])
            r = rng.uniform(0.3, 1.0)
            k = int(rng.integers(0, 2))
            c2 = c.copy()
            c2[k] += 0.5 * r
            ids = [None, None]
            for j in ((0, 1) if first == 0 else (1, 0)):
                ids[j] = w.sphere(c if j == 0 else c2, r, j)
            o = rng.uniform(-0.3, 0.3, 3).astype(np.float32)
            a1 = (np.asarray(w.spheres[ids[0]][0]) - o).astype(np.float32)
            a2 = (np.asarray(w.spheres[ids[1]][0]) - o).astype(np.float32)
            fams.append((_ray(o, a1), 4 + k, a1[k], a2[k], None))
    for n, (x, y) in enumerate(((6.0, 1.0), (-6.0, -1.0), (6.0, -3.0), (-6.0, 3.0))):
        q = (x, y, -4.5)                                                   # small: front at z = -4
        p = (x, y, -5.0)                                                   # large: front at z = -4
        if n % 2 == 0:
            w.sphere(q, 0.5, 0); w.sphere(p, 1.0, 1)
        else:
            w.sphere(p, 1.0, 1); w.sphere(q, 0.5, 0)
        for z0 in (0.0, 1.0, -1.0, 0.5, -2.0):
            for s in (1.0, 0.25, 8.0):
                extra.append(_ray((x, y, z0), (0.0, 0.0, -s)))
        o = np.array([x, y, 0.0], np.float32)
        for k, sgn in ((0, 1.0), (0, -1.0), (1, 1.0), (1, -1.0)):
            fams.append((_ray(o, (0.0, 0.0, -1.0)), k, F(o[k]), F(o[k] + sgn * 0.2), None))
            fams.append((_ray(o, (0.0, 0.0, -1.0)), 4 + k, F(0.0), F(sgn * 0.03), None))
    return w, fams, extra


def regime_direct_ties(huge, out_of_range_first):
    """One DIRECT group with a tie between a sphere whose discriminant is outside [2^-100, 2^100] (finished by the
    group's second pass) and one inside it.  huge: radii 2^51 (disc 2^102) and 2^49 (disc 2^98), both fronts at
    t = 2^50 on the axis ray; tiny: a sphere of radius 2^-60 whose axis-ray discriminant rounds to 0 at t = 1 and a unit
    sphere with its front at t = 1."""
    w = World()
    if huge:
        spheres = [((0.0, 0.0, -3.0 * 2.0 ** 50), 2.0 ** 51), ((0.0, 0.0, -3.0 * 2.0 ** 49), 2.0 ** 49)]
    else:
        spheres = [((0.0, 0.0, -1.0), 2.0 ** -60), ((0.0, 0.0, -2.0), 1.0)]
    w.sphere((5.0, 5.0, 5.0), 0.5, 3)
    for j in ((0, 1) if out_of_range_first else (1, 0)):
        w.sphere(spheres[j][0], spheres[j][1], j)
    w.sphere((-5.0, 5.0, 5.0), 0.5, 3)
    fams, extra = [], []
    for s in (1.0, 2.0 ** -10, 2.0 ** 20, 3.0):
        extra.append(_ray((0.0, 0.0, 0.0), (0.0, 0.0, -s)))
        extra.append(_ray((0.0, 0.0, 0.0), (0.0, 0.0, -s), t_max=F(2.0 ** 50 if huge else 1.0)))
    if huge != out_of_range_first:
        # the axis tie goes to the sphere that loses just off the axis (the larger one is nearer there): a crossing.
        # In the other two orders the same sphere wins on and off the axis, and the axis rays carry the tie alone.
        for k in (4, 5):
            for hi in (1e-3, -1e-3, 0.3, -0.3):
                fams.append((_ray((0.0, 0.0, 0.0), (0.0, 0.0, -1.0)), k, F(0.0), F(hi), None))
    return w, fams, extra


def regime_triangle_parallel(rng):
    """Rays nearly parallel to a big triangle's plane: den = n.dir crosses -+1e-8.  The reference's plane term is
    t = (n.o + n.v0) / den (sic, common.rs:140), so with the plane z = z0 an origin at z = -z0 + h puts the hit at
    t = h / d.z."""
    w = World()
    fams = []
    for k, size in enumerate((1.0, 30.0, 100.0)):
        z = -float(k) * 3.0
        w.triangle((-size, -size, z), (size, -size, z), (0.0, size, z), k % 4)
        A = 4.0 * size * size                                              # |n| of the triangle
        for _ in range(6):
            th = rng.uniform(0, 2 * np.pi)
            for side in (1.0, -1.0):
                dz = 1e-8 / A                                              # |d.z| where |den| = 1e-8
                h = F(side * 0.2 * size * dz)
                o = np.array([rng.uniform(-0.2, 0.2) * size, rng.uniform(-0.3, 0.0) * size, -z + h], np.float32)
                a = np.array([np.cos(th), np.sin(th), 0.0], np.float32)
                fams.append((_ray(o, a), 6, F(side * dz * 10.0), F(side * dz * 0.1), None))
    return w, fams, []


def _tri_frame(v0, v1, v2):
    v0, v1, v2 = (np.asarray(v, np.float64) for v in (v0, v1, v2))
    return v0, v1, v2, np.cross(v1 - v0, v2 - v0)


def _aim(o, pt, v0, n):
    """The direction from o whose reference hit is the triangle point pt: t = (n.o + n.v0) / n.d puts the hit on the
    plane n.x = n.v0 + 2 n.o, which the inside tests project along n onto the triangle."""
    return pt + n * (2.0 * (n @ o) / (n @ n)) - o


def _slide(a, n, out):
    """(component k, displacement of the hit point along `out` per unit of a[k]) of the direction component that moves
    the hit most across an edge."""
    g = np.array([(np.eye(3)[k] - a * n[k] / (n @ a)) @ out for k in range(3)])
    k = int(np.argmax(np.abs(g)))
    return k, g[k]


def regime_triangle_window(rng):
    """t = 0.001 (origin slid along the ray), t = t_max, two triangles at adjacent t in both list orders, duplicate
    triangles, and a sphere and a triangle at the same t (the triangle's window is inclusive)."""
    w = World()
    fams, extra = [], []
    for k in range(6):
        P0 = rng.uniform(-1, 1, 3) * 10.0 ** rng.uniform(0, 2)
        s = 10.0 ** rng.uniform(-1, 0.5)
        j = w.triangle(*[P0 + rng.uniform(-1, 1, 3) * s for _ in range(3)], m=k % 4)
        v0, v1, v2, n = _tri_frame(*w.triangles[j][:3])
        nh = n / np.linalg.norm(n)
        cen = (v0 + v1 + v2) / 3.0
        d = _unit(rng)
        if abs(d @ nh) < 0.3:
            d = d + nh
        d /= np.linalg.norm(d)
        # an origin whose hit is at t0 = 0.002 over the centroid; moving it by x e_k moves t by x n_k / n.d
        t0 = 0.002
        plane = lambda x: x - nh * (nh @ x)                                # noqa: E731
        o = plane(cen) - t0 * plane(d) + nh * (t0 * (n @ d) - n @ v0) / np.linalg.norm(n)
        kk = int(np.argmax(np.abs(n)))
        for t_lo, t_hi in ((0.0005, 0.004), (0.004, 0.0005)):
            x = lambda t: (t - t0) * (n @ d) / n[kk]                      # noqa: E731
            fams.append((_ray(o.astype(np.float32), d), kk, F(o[kk] + x(t_lo)), F(o[kk] + x(t_hi)), None))
        o = (cen - d * rng.uniform(1, 5)).astype(np.float32)
        a = _aim(o.astype(np.float64), cen, v0, n).astype(np.float32)
        fams.append((_ray(o, a), 3, F(0.0011), F(1e6), None))             # t_max across the hit's t
    for first in (0, 1):                                                   # crossing planes z = -3 and z = -3 + (x - x0)/8
        x0 = 10.0 * (first * 2 - 1)
        flat = ((x0 - 2, -2, -3.0), (x0 + 2, -2, -3.0), (x0, 2, -3.0))
        tilt = ((x0 - 2, -2, -3.25), (x0 + 2, -2, -2.75), (x0, 2, -3.0))
        for j in ((0, 1) if first == 0 else (1, 0)):
            w.triangle(*(flat if j == 0 else tilt), m=j)
        for _ in range(4):                                                 # from the world's origin: n.o = 0
            a = np.array([x0, rng.uniform(-0.5, 0.5), -3.0], np.float32)
            fams.append((_ray((0.0, 0.0, 0.0), a), 4, F(x0 - 0.5), F(x0 + 0.5), None))
    dup = ((20.0, -2.0, -4.0), (24.0, -2.0, -4.5), (22.0, 2.0, -4.25))
    w.triangle(*dup, m=0)
    w.triangle(*dup, m=3)
    for _ in range(6):
        a = np.array([22.0 + rng.uniform(-0.5, 0.5), rng.uniform(-0.5, 0.5), -4.25], np.float32)
        extra.append(_ray((0.0, 0.0, 0.0), a))
        fams.append((_ray((0.0, 0.0, 0.0), a), 4, a[0], F(30.0), None))
        fams.append((_ray((0.0, 0.0, 0.0), a), 5, a[1], F(-3.0), None))
    # a sphere and a triangle through the same point at t = 4 on the ray from (x, 0, 0) along -z; the plane tilts
    # 1/16 in y (n = (0, 1, 16): n.o = 0), so just above the axis the sphere is nearer and just below the triangle
    x = 40.0
    w.sphere((x, 0.0, -5.0), 1.0, 1)
    w.triangle((x - 2, -2, -4 + 0.125), (x + 2, -2, -4 + 0.125), (x, 2, -4 - 0.125), m=0)
    for t_max in (INF, 4.0, float(np.nextafter(F(4.0), F(-INF))), float(np.nextafter(F(4.0), F(INF)))):
        for s in (1.0, 2.0, 0.125):
            extra.append(_ray((x, 0.0, 0.0), (0.0, 0.0, -s), t_max))
    for hi in (0.05, -0.05):
        fams.append((_ray((x, 0.0, 0.0), (0.0, 0.0, -1.0)), 5, F(0.0), F(hi), None))
    return w, fams, extra


def _k_of(v0, v1, v2):
    """K of rt_scene.cpp triangle_cull_record (the edge stage runs when |o|_1 + t < K); -inf when never."""
    v0, v1, v2 = (np.asarray(v, np.float64) for v in (v0, v1, v2))
    n = np.cross(v1 - v0, v2 - v0)
    nn = n @ n
    if not (nn > 0) or not np.isfinite(nn):
        return -INF
    lmax = np.sqrt(max((v1 - v0) @ (v1 - v0), (v2 - v1) @ (v2 - v1), (v0 - v2) @ (v0 - v2)))
    K = 4096.0 * np.sqrt(nn) / lmax - max(np.abs(v0).sum(), np.abs(v1).sum(), np.abs(v2).sum())
    return K if K > 0 and np.isfinite(K) else -INF


def regime_edges(rng):
    """Each edge and each vertex of regular, large, needle and distant triangles crossed by a turning direction, from
    origins near (the edge stage decides: |o|_1 + t < K) and far (the K fallback).  Needle, distant and remote (size 0.5 at
    10^6) triangles have K = -inf: the edge stage never rejects them."""
    w = World()
    fams = []
    kinds = (("regular", 1.0, 3.0), ("large", 50.0, 20.0), ("needle", 3.0, 4.0), ("distant", 5.0, 2.0e4),
             ("remote", 0.5, 1.0e6))
    for m, (kind, size, dist) in enumerate(kinds):
        for rep in range(2):
            ctr = _unit(rng) * dist
            ctr[2] = -abs(ctr[2]) - 1.0
            v = [ctr + rng.uniform(-1, 1, 3) * size for _ in range(3)]
            if kind == "needle":
                v[2] = v[0] + (v[1] - v[0]) * 0.5 + rng.uniform(-1, 1, 3) * 1e-4 * size
            j = w.triangle(*v, m=m)
            v0, v1, v2, n = _tri_frame(*w.triangles[j][:3])
            nh = n / np.linalg.norm(n)
            V = (v0, v1, v2)
            cen = (v0 + v1 + v2) / 3.0
            K = _k_of(v0, v1, v2)
            for e in range(6):
                if e < 3:                                                  # edge e: V[e] -> V[e+1]
                    a_, b_ = V[e], V[(e + 1) % 3]
                    pt = a_ + (b_ - a_) * rng.uniform(0.2, 0.8)
                    out = np.cross(nh, (b_ - a_) / np.linalg.norm(b_ - a_))
                    if out @ (cen - pt) > 0:
                        out = -out
                else:                                                      # vertex e - 3, away from the centroid
                    pt = V[e - 3]
                    out = pt - cen
                    out -= nh * (nh @ out)
                    out /= np.linalg.norm(out)
                h = max(abs((cen - pt) @ out), 1e-12)
                for L in (0.5 * dist + 1.0, 3.0 * K if K > 0 else 1e3 * dist):
                    d = _unit(rng)
                    if abs(d @ nh) < 0.4:
                        d = d - nh * np.sign(d @ nh or 1.0)
                    d /= np.linalg.norm(d)
                    o = (pt - d * L).astype(np.float32)
                    if np.max(np.abs(o)) > 2.0 ** 40:
                        continue
                    a = _aim(o.astype(np.float64), pt, v0, n)
                    k, g = _slide(a, n, out)
                    if abs(g) < 1e-6:
                        continue
                    reach = float(np.abs(o).sum()) + float(np.linalg.norm(a))
                    a = a.astype(np.float32)
                    for f in (0.5, 0.05):
                        fams.append((_ray(o, a), 4 + k, F(a[k] - f * h / g), F(a[k] + f * h / g), ("edge", kind, reach < K)))
    return w, fams, []


def regime_edges_far(rng):
    """Unit-sized triangles in planes z = const seen from origins far past K (|o| = 2^23 to 2^40, 2^40 the domain's
    limit, in every direction): hits aimed inside them, and crossings of each edge and vertex.  There the approximate barycentrics of
    the edge stage are off by more than its half-height margin, so only the K fallback keeps the stage from rejecting
    these hits."""
    w = World()
    fams, extra = [], []
    tris = []
    for k, (z, sc, dx) in enumerate(((-3.0, 1.0, 0.0), (-5.0, 2.0, 1.5), (-3.5, 0.5, -2.0), (-8.0, 1.0, 0.25))):
        tris.append(w.triangle((dx - 0.5 * sc, -0.5 * sc, z), (dx + 0.5 * sc, -0.5 * sc, z), (dx, 0.5 * sc, z), m=k % 4))
    for j in tris:
        v0, v1, v2, n = _tri_frame(*w.triangles[j][:3])
        nh = n / np.linalg.norm(n)
        V = (v0, v1, v2)
        cen = (v0 + v1 + v2) / 3.0
        for e2 in range(23, 41):
            o = (_unit(rng) * 2.0 ** e2).astype(np.float32)
            o64 = o.astype(np.float64)
            for _ in range(3):                                            # hits aimed inside
                b = rng.dirichlet((2.0, 2.0, 2.0))
                extra.append(_ray(o, _aim(o64, b[0] * v0 + b[1] * v1 + b[2] * v2, v0, n).astype(np.float32)))
            e = int(rng.integers(0, 3))                                    # one edge and one vertex per origin
            for pt in (V[e] + (V[(e + 1) % 3] - V[e]) * rng.uniform(0.2, 0.8), V[e]):
                out = pt - cen
                out -= nh * (nh @ out)
                h = np.linalg.norm(out)
                a = _aim(o64, pt, v0, n)
                k, g = _slide(a, n, out / h)
                if abs(g) < 1e-6:
                    continue
                af = a.astype(np.float32)
                fams.append((_ray(o, af), 4 + k, F(a[k] - 0.5 * h / g), F(a[k] + 0.5 * h / g), ("edge", "unit-far", False)))
    return w, fams, extra


def regime_cull_bound(rng):
    """Tight groups (8 spheres in a ball of radius 0.5) and loose ones (spheres spread over 40 units): tangencies of
    their members from near and far origins, and from origins with o.o just above and below 2^-126 (below, the CULL
    walk hands the ray to the FILTER walk)."""
    w = World()
    for g in range(5):
        ctr = np.array([rng.uniform(-8, 8), rng.uniform(-4, 4), rng.uniform(-12, -6)])
        for _ in range(8):
            w.sphere(ctr + _unit(rng) * rng.uniform(0, 0.4), rng.uniform(0.05, 0.2), int(rng.integers(0, 4)))
    for _ in range(34):
        w.sphere((rng.uniform(-20, 20), rng.uniform(-20, 20), rng.uniform(-40, -2)), rng.uniform(0.05, 0.3),
                 int(rng.integers(0, 4)))
    fams = []
    members = list(rng.permutation(len(w.spheres))[:20])
    near = [rng.uniform(-0.5, 0.5, 3) for _ in range(2)]
    _tangency_families(rng, w, members, near, fams)
    far = []
    for L in (1e3, 1e5, 1e7):
        v = _unit(rng)
        v[2] = abs(v[2])
        far.append(v * L)
    _tangency_families(rng, w, members[:10], far, fams)
    s = F(2.0 ** -63)
    tiny = [(s, 0, 0), (np.nextafter(s, F(0)), 0, 0), (np.nextafter(s, F(1)), 0, 0), (0, -s, 0),
            (0, 0, np.nextafter(s, F(0))), (F(2.0 ** -63.5), F(2.0 ** -63.5), 0), (F(1e-30), 0, 0)]
    _tangency_families(rng, w, members[:8], [np.array(t, np.float32) for t in tiny], fams)
    return w, fams, []


def regime_cull_ties(rng):
    """Nested spheres touching at their fronts, at exact ties on axis rays, placed so that the CULL walk visits the
    one with the larger list index first: a large sphere (an "always" group, visited before the others) after its
    small partner, and a pair of small spheres whose spatial order is the reverse of the list order; plus duplicate
    spheres with different materials.  Over 64 spheres, so every walk applies."""
    w = World()
    for i in range(64):
        w.sphere((-12.0 + 0.375 * i, -3.0, -6.0 + 0.03125 * (i % 5)), 0.125, i % 4)
    fams, extra = [], []
    axis = []
    for n, x in enumerate((-9.0, -6.0, -3.0, 3.0, 6.0, 9.0)):
        y = 1.0 if n % 2 else 3.0
        if n < 4:                     # small (r 0.5, z -4.5) and large (r 1, z -5: above 8x the median radius)
            small, large = ((x, y, -4.5), 0.5), ((x, y, -5.0), 1.0)
        else:                         # two small ones: r 0.25 at z -4.25 and r 0.5 at z -4.5 (lower Morton key)
            small, large = ((x, y, -4.25), 0.25), ((x, y, -4.5), 0.5)
        order = (small, large) if n % 3 != 2 else (large, small)
        for m, (c, r) in enumerate(order):
            w.sphere(c, r, m)
        axis.append((x, y))
    for x, y in ((0.0, -1.0), (12.0, -1.0)):                                # duplicates
        w.sphere((x, y, -5.0), 0.5, 0)
        w.sphere((x, y, -5.0), 0.5, 1)
        axis.append((x, y))
    for x, y in axis:
        for z0 in (0.0, 1.0, -1.0, 0.5):
            for s in (1.0, 4.0):
                extra.append(_ray((x, y, z0), (0.0, 0.0, -s)))
        o = np.array([x, y, 0.0], np.float32)
        for k, sgn in ((0, 1.0), (0, -1.0), (1, 1.0), (1, -1.0)):
            fams.append((_ray(o, (0.0, 0.0, -1.0)), k, F(o[k]), F(o[k] + sgn * 0.2), None))
            fams.append((_ray(o, (0.0, 0.0, -1.0)), 4 + k, F(0.0), F(sgn * 0.05), None))
    return w, fams, extra


# name -> (builder, decision, minimum pairs)
REGIMES = {
    "tangent_unit":      (lambda rng: regime_tangent_unit(rng), "sphere disc >= 0", 40),
    "tangent_negative":  (lambda rng: regime_tangent_unit(rng, negative=True), "sphere disc >= 0", 40),
    "tangent_ground":    (regime_tangent_ground, "sphere disc >= 0", 20),
    "tangent_far":       (regime_tangent_far, "sphere disc >= 0", 20),
    "tangent_big_c":     (regime_tangent_big_c, "sphere disc >= 0", 20),
    "root_choice":       (regime_root_choice, "root1 > 0.001, t > 0.001", 30),
    "sphere_window":     (regime_sphere_window, "t < closest", 15),
    # direct_huge_out and direct_tiny_in are tie-only sets: no crossing, their axis rays carry the tie
    "direct_huge_out":   (lambda rng: regime_direct_ties(True, True), "t < closest (second pass)", 0),
    "direct_huge_in":    (lambda rng: regime_direct_ties(True, False), "t < closest (second pass)", 4),
    "direct_tiny_out":   (lambda rng: regime_direct_ties(False, True), "t < closest (second pass)", 4),
    "direct_tiny_in":    (lambda rng: regime_direct_ties(False, False), "t < closest (second pass)", 0),
    "triangle_parallel": (regime_triangle_parallel, "|den| < 1e-8", 8),
    "triangle_window":   (regime_triangle_window, "t >= 0.001, t <= t_max, t < best", 20),
    "edges":             (regime_edges, "edge tests", 60),
    "edges_far":         (regime_edges_far, "edge tests, K fallback", 8),
    "cull_bound":        (regime_cull_bound, "CULL bound, tiny origins", 300),
    "cull_ties":         (regime_cull_ties, "t < closest (CULL)", 20),
}
TANGENT_REGIMES = ("tangent_unit", "tangent_negative", "tangent_ground", "tangent_far", "tangent_big_c", "cull_bound")

_SETS = {}


def boundary_set(ob, name):
    """{world, text, cam, pairs [m, 2, 8], tags, rays (pairs then extras)} of a regime, built once per process."""
    if name not in _SETS:
        builder, _, _ = REGIMES[name]
        rng = np.random.default_rng(list(REGIMES).index(name) * 7919 + 11)
        w, fams, extra = builder(rng)
        text, cam, world = parse_exact(ob, w)
        pairs, tags = bisect(ob, world, fams)
        rays = np.concatenate([pairs.reshape(-1, 8)] + ([np.array(extra, np.float32)] if extra else []))
        _SETS[name] = dict(w=w, world=world, text=text, cam=cam, pairs=pairs, tags=tags, rays=rays)
    return _SETS[name]


def exact_disc(o, c, r, a):
    """The reference's discriminant (oc.d)^2 - (oc.oc - r^2) in exact arithmetic from the float32 origin, centre,
    radius and the float32 normalised direction; and Q = o.o + c.c + r^2."""
    d = test_rays.npo.nvec(*(F(x) for x in a))
    o, c, d, r = [Fraction(float(x)) for x in o], [Fraction(float(x)) for x in c], [Fraction(float(x)) for x in d], \
        Fraction(float(r))
    oc = [o[i] - c[i] for i in range(3)]
    hb = sum(oc[i] * d[i] for i in range(3))
    D = hb * hb - (sum(x * x for x in oc) - r * r)
    return D, sum(x * x for x in o) + sum(x * x for x in c) + r * r


# ----------------------------------------------------------------------------------------------- generator coverage

@pytest.mark.parametrize("name", list(REGIMES))
def test_boundary_pairs_straddle_their_decision(ob, name):
    """Every pair is two rays one float apart whose records differ, by the reference and by the literal restatement;
    the regime yields its stated number of pairs."""
    s = boundary_set(ob, name)
    pairs = s["pairs"]
    assert len(pairs) >= REGIMES[name][2], f"{name}: {len(pairs)} pairs"
    if len(pairs):
        diff = pairs[:, 0] != pairs[:, 1]
        assert (diff.sum(axis=1) == 1).all()
        ka, kb = keys(pairs[:, 0][diff]), keys(pairs[:, 1][diff])
        assert (np.abs(ka - kb) == 1).all()
        want = reference(ob, s["world"], s["rays"])
        n = len(pairs)
        assert _differ(want, want, slice(0, 2 * n, 2), slice(1, 2 * n, 2)).all()
    assert_same(literal_records(s["world"], s["rays"]), reference(ob, s["world"], s["rays"]))


def test_tangent_pairs_sit_inside_the_filter_margin(ob):
    """The exact discriminant of the crossed sphere, from the float32 inputs, on both rays of a tangency pair: many
    pairs have |D| <= 64u Q on both rays (Q = o.o + c.c + r^2), with both signs of D among them — the rays sit inside
    the FILTER walk's 128u margin, not outside it."""
    total, signs = 0, set()
    for name in TANGENT_REGIMES:
        s = boundary_set(ob, name)
        inside = 0
        for pair, tag in zip(s["pairs"], s["tags"]):
            if tag is None:
                continue
            c, r, _ = s["w"].spheres[tag]
            Ds = [exact_disc(ray[0:3], c, r, ray[4:7]) for ray in pair]
            if all(abs(D) <= 64 * U * Q for D, Q in Ds):
                inside += 1
                signs.update(np.sign(float(D)) for D, _ in Ds)
        assert inside >= 5, f"{name}: {inside} pairs within 64u Q of the tangent"
        total += inside
    assert total >= 100 and {-1.0, 1.0} <= signs


def test_edge_pairs_cover_both_sides_of_the_k_fallback(ob):
    s = boundary_set(ob, "edges")
    near = [t[2] for t in s["tags"] if t is not None]
    kinds = {t[1] for t in s["tags"] if t is not None}
    assert sum(near) >= 20 and len(near) - sum(near) >= 20 and kinds == {"regular", "large", "needle", "distant", "remote"}


def test_far_origins_hit_unit_triangles(ob):
    """The far-origin set is mostly hits, from every octave of |o| between 2^23 and 2^40: rays the edge stage would
    wrongly reject without its K fallback."""
    s = boundary_set(ob, "edges_far")
    n = 2 * len(s["pairs"])
    rays = s["rays"][n:]
    rec = reference(ob, s["world"], rays)
    hit = rec["prim"] >= 0
    assert hit.sum() >= 150
    octaves = np.floor(np.log2(np.linalg.norm(rays[hit][:, 0:3].astype(np.float64), axis=1)))
    assert set(octaves.astype(int)) >= set(range(23, 40))


def test_direct_tie_worlds_put_an_out_of_range_discriminant_in_a_tie(ob):
    """The axis ray of the DIRECT tie worlds ties two spheres of one group, and the one whose discriminant is outside
    [2^-100, 2^100] wins exactly when it comes first in the list (sphere 1; sphere 0 is elsewhere)."""
    for huge in (True, False):
        for first in (True, False):
            s = boundary_set(ob, f"direct_{'huge' if huge else 'tiny'}_{'out' if first else 'in'}")
            rec = reference(ob, s["world"], _rays([0.0, 0.0, 0.0], [0.0, 0.0, -1.0]))
            assert rec["depth"][0] == F(2.0 ** 50 if huge else 1.0)
            assert rec["prim"][0] == 1, (huge, first, rec["prim"][0])
            assert (abs(s["w"].spheres[1][1]) == F(2.0 ** 51 if huge else 2.0 ** -60)) == first


def test_cull_ties_are_visited_against_list_order(ob):
    """On the CULL tie world, the large sphere of a nested pair sits in an "always" group and the small pairs are in
    the reverse Morton order, so some winning tie partners are visited second by the CULL walk."""
    s = boundary_set(ob, "cull_ties")
    rec = reference(ob, s["world"], s["rays"])
    spheres = s["w"].spheres
    axis = [i for i, r in enumerate(s["rays"]) if r[4] == 0 and r[5] == 0 and rec["prim"][i] >= 64
            and spheres[rec["prim"][i]][0][:2] == (r[0], r[1])]
    assert len(axis) >= 20
    later = 0
    for i in axis:
        p = rec["prim"][i]
        twin = [j for j in range(64, len(spheres)) if j != p and spheres[j][0][:2] == spheres[p][0][:2]]
        assert len(twin) == 1 and twin[0] > p                             # the tie goes to the lower index
        later += abs(spheres[twin[0]][1]) > abs(spheres[p][1]) or spheres[twin[0]][0][2] < spheres[p][0][2]
    assert later >= 8


# ------------------------------------------------------------------------------------------ device functions on host

@pytest.fixture(scope="module")
def ray_libs():
    return test_rays._load_hostsim("librays_hostsim.so"), test_rays._load_hostsim("librays_hostsim_perturb.so")


@pytest.fixture(scope="module")
def occ_libs():
    return (test_occlusion._load_hostsim("libocclusion_hostsim.so"),
            test_occlusion._load_hostsim("libocclusion_hostsim_perturb.so"))


def _host_worlds(ob, s):
    """(text, oracle world, walks) of the set's world as built, and padded past 64 spheres for the FILTER and CULL
    walks when it is smaller."""
    out = [(s["text"], s["world"], (DIRECT, FILTER) + ((CULL,) if len(s["w"].spheres) >= FILTER_FROM else ()))]
    n = s["w"].n_fill_wide()
    if n:
        text, _, world = parse_exact(ob, s["w"], n)
        out.append((text, world, (DIRECT, FILTER, CULL)))
    return out


@pytest.mark.parametrize("name", list(REGIMES))
def test_ray_hit_on_host(ob, ray_libs, name):
    s = boundary_set(ob, name)
    for text, world, walks in _host_worlds(ob, s):
        want = reference(ob, world, s["rays"])
        for L in ray_libs:
            for walk in walks:
                got = test_rays._hostsim(L, text, s["rays"], walk)
                assert_same(got, want)


@pytest.mark.parametrize("name", list(REGIMES))
def test_ray_occluded_on_host(ob, occ_libs, name):
    s = boundary_set(ob, name)
    rays = np.concatenate([s["rays"], _t_max_variants(ob, s["world"], s["rays"])])
    for text, world, walks in _host_worlds(ob, s):
        want = test_occlusion.expected(ob, world, rays)
        for L in occ_libs:
            for walk in walks:
                test_occlusion.assert_answers(test_occlusion._hostsim(L, text, rays, walk), want)


def _t_max_variants(ob, world, rays):
    """The set's rays with t_max at their hit's t and one float either side: the any-hit walk's window edges."""
    rec = reference(ob, world, rays)
    hit = rec["prim"] >= 0
    out = []
    for f in (lambda t: t, lambda t: np.nextafter(t, F(-INF)), lambda t: np.nextafter(t, F(INF))):
        r = rays[hit].copy()
        r[:, 3] = f(rec["depth"][hit])
        out.append(r)
    return np.concatenate(out)


# ------------------------------------------------------------------------------------------------------ tie worlds

def tie_world(wide):
    """Duplicate spheres and triangles with different materials, nested spheres touching at their fronts in both list
    orders, and a sphere and a triangle meeting at one point, in front of the camera.  wide: over 64 spheres (FILTER
    and CULL walks), else under (DIRECT)."""
    w = World()
    rng = np.random.default_rng(404)
    if wide:
        for i in range(60):
            w.sphere((-6.0 + 0.2 * i, -2.0 + 0.1 * (i % 3), -6.0 - 0.125 * (i % 4)), 0.09, i % 4)
    for n, x in enumerate((-2.0, -1.0, 0.0, 1.0, 2.0)):
        small, large = ((x, 0.5, -4.5), 0.25), ((x, 0.5, -4.75), 0.5)
        for m, (c, r) in enumerate((small, large) if n % 2 else (large, small)):
            w.sphere(c, r, m + 1)
        w.sphere((x, -0.5, -4.0), 0.3, n % 4)
        w.sphere((x, -0.5, -4.0), 0.3, (n + 2) % 4)
    w.sphere((0.0, -100.5, -4.0), 100.0, 0)
    for k in range(3):
        v = [np.array([rng.uniform(-2.5, 2.5), rng.uniform(0.8, 1.5), -3.5]) + rng.uniform(-0.6, 0.6, 3) for _ in range(3)]
        w.triangle(*v, m=k % 4)
        w.triangle(*v, m=(k + 1) % 4)
    w.sphere((2.5, -1.2, -5.0), 1.0, 4)
    w.triangle((0.5, -3.2, -4.0 + 0.125), (4.5, -3.2, -4.0 - 0.125), (2.5, 0.8, -4.0), m=2)
    return w


TIE_FRAME = (48, 32, 2, 6)          # W, H, spp, depth


def _tie(ob, wide):
    w = tie_world(wide)
    text, cam, world = parse_exact(ob, w)
    assert (len(w.spheres) >= FILTER_FROM) == wide
    return text, cam, world


@pytest.fixture(scope="module")
def render_host():
    import test_hostsim
    return test_hostsim._load("libhostsim.so")


@pytest.mark.parametrize("wide", [False, True], ids=["under64", "over64"])
def test_tie_worlds_render_on_host(ob, render_host, wide):
    text, cam, world = _tie(ob, wide)
    W, H, spp, depth = TIE_FRAME
    want, rays, _ = ob.ray_trace(world, cam, W, H, spp, depth, fixed_jitter=True)
    cf = cam.floats()
    for flags in ((DIRECT, FILTER, CULL, NP2) if wide else (DIRECT, FILTER)):
        out = np.zeros((H, W, 4), np.uint8)
        n = C.c_uint64()
        rc = render_host.hostsim_render(text.encode(), cf.ctypes.data_as(C.POINTER(C.c_float)), W, H, spp, depth,
                                        ob.SEED_DEFAULT, flags | 1, 0, 0, out.ctypes.data, C.byref(n))   # bit 0: fixed jitter
        assert rc == 0 and n.value == rays, (hex(flags), n.value, rays)
        assert np.array_equal(out, want), f"walk {flags:#x}: {int((out != want).any(axis=2).sum())} pixels differ"


# ------------------------------------------------------------------------------------------------------------ GPU

def _gpu_worlds(ob, s):
    """(label, text, oracle world, expected launch statistics by cull flag) of a set: as built (DIRECT under 64
    spheres), padded past 64 spheres (FILTER / CULL, staged in shared memory) and past shared memory (global)."""
    out = []
    n = len(s["w"].spheres)
    if n < FILTER_FROM:
        out.append(("direct", s["text"], s["world"], {c: dict(filtered=0, culled=0, resident=1) for c in (False, True)}))
    fill = s["w"].n_fill_wide()
    text, _, world = parse_exact(ob, s["w"], fill) if fill else (s["text"], None, s["world"])
    out.append(("smem", text, world, {c: dict(filtered=1, culled=int(c), resident=1) for c in (False, True)}))
    text, _, world = parse_exact(ob, s["w"], s["w"].n_fill_global())
    out.append(("global", text, world, {c: dict(filtered=1, culled=int(c), resident=0, smem_bytes=0) for c in (False, True)}))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(REGIMES))
def test_gpu_ray_and_occlusion_kernels(gpu_rt, ob, name):
    s = boundary_set(ob, name)
    rays = np.concatenate([s["rays"], _t_max_variants(ob, s["world"], s["rays"])])
    for label, text, world, stats in _gpu_worlds(ob, s):
        h = gpu_rt.load_world(text)
        want = reference(ob, world, rays)
        want_occ = test_occlusion.answers(want["prim"])
        for cull in (False, True):
            st = gpu_rt.RenderStats()
            assert_same(test_rays._gpu(gpu_rt, h, rays, cull, st), want, canonical_nan=True)
            got = {k: int(getattr(st, k)) for k in stats[cull]}
            assert got == stats[cull] and st.rays == len(rays), (label, cull, got)
            st = gpu_rt.RenderStats()
            test_occlusion.assert_answers(test_occlusion._gpu(gpu_rt, h, rays, cull, st), want_occ)
            got = {k: int(getattr(st, k)) for k in stats[cull]}
            assert got == stats[cull], (label, cull, got)


def check_tie_render(rt, ob, wide, cull, paths_per_lane=1):
    """The exact render of a tie world: RGBA8, ray count and the float4 colour sums against the oracle, and the launch
    statistics of the walk it must take."""
    import torch
    text, cam, world = _tie(ob, wide)
    W, H, spp, depth = TIE_FRAME
    want, rays, want_acc = ob.ray_trace(world, cam, W, H, spp, depth, fixed_jitter=True, want_accum=True)
    h = rt.load_world(text)
    fb, st = rt.Framebuffer(W, H), rt.RenderStats()
    rt.render_with_options(fb, h, rt.Options(spp, depth, fixed_jitter=True, group_cull=cull), st)
    walk = dict(filtered=int(wide), culled=int(wide and cull), paths_per_lane=paths_per_lane)
    assert {k: int(getattr(st, k)) for k in walk} == walk, (wide, cull, st.filtered, st.culled, st.paths_per_lane)
    assert st.rays == rays, (st.rays, rays)
    got = fb.pixels.copy()
    assert np.array_equal(got, want), f"{int((got != want).any(axis=2).sum())} pixels differ from the oracle"
    accum = torch.full((H, W, 4), 7.0, dtype=torch.float32, device="cuda")
    out = torch.zeros((H, W), dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    st = rt.RenderStats()
    rt.render_device(h, rt.Options(spp, depth, fixed_jitter=True, accum_out=True, group_cull=cull), W, H,
                     out.data_ptr(), accum.data_ptr(), 0, st)
    assert st.rays == rays
    acc = accum.cpu().numpy()
    bad = np.argwhere(acc.view(np.uint32) != np.asarray(want_acc, np.float32).view(np.uint32))
    assert bad.size == 0, f"{len(bad)} float4 sums differ, first at {bad[0].tolist()}"
    assert np.array_equal(out.cpu().numpy().view(np.uint8).reshape(H, W, 4), want)


@pytest.mark.gpu
@pytest.mark.parametrize("wide,cull", [(False, False), (True, False), (True, True)], ids=["DIRECT", "FILTER", "CULL"])
def test_gpu_tie_world_render(gpu_rt, ob, wide, cull):
    check_tie_render(gpu_rt, ob, wide, cull)


@pytest.mark.gpu
def test_gpu_tie_world_render_two_paths_per_lane(gpu_rt):
    """The FILTER walk with two paths per lane (RT_PATHS_PER_LANE is read once per process: a subprocess)."""
    code = ("import sys, traceback\n"
            f"sys.path[:0] = [{str(ROOT)!r}, {str(ROOT / 'oracle')!r}, {str(HERE)!r}]\n"
            "import importlib, oracle_binding as ob, test_boundary_rays as m\n"
            "rt = importlib.import_module('rust-swift-raytracer_b200')\n"
            "try:\n    m.check_tie_render(rt, ob, True, False, paths_per_lane=2); print('RESULT ok')\n"
            "except AssertionError:\n    print('RESULT ' + traceback.format_exc(limit=3).replace(chr(10), ' | '))\n")
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=900,
                       env=dict(os.environ, RT_PATHS_PER_LANE="2"), cwd=str(ROOT))
    lines = [l for l in r.stdout.splitlines() if l.startswith("RESULT ")]
    assert r.returncode == 0 and lines, r.stdout[-4000:] + r.stderr[-4000:]
    assert lines[-1] == "RESULT ok", lines[-1]
