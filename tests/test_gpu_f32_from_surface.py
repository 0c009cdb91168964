"""The f32 traversal (k_f_trace6) query by query on rays that start on a surface, against the f64 classifier.

Bounce 0 runs the id-exact kernel and is the only bounce whose rays have no source primitive.  Every ray k_f_trace6
traces in a fast frame -- bounces >= 1 and shadow rays -- starts on the primitive it just left, and leaf_f3 applies the
source rules to it: a source triangle or Rect is never re-hit, a source sphere is skipped when the ray leaves it and
re-entered at the far root (or the chord -2 hb) when the ray goes in (DESIGN.md 4.3).  tests/native/brute_hit.c
classifies each (ray, primitive) pair with those rules at margins derived from the kernel's f32 roundings (its header
states them), and on rays whose answer does not depend on rounding the kernel must return the f64 answer exactly.

The CPU tests check the source rules of the classifier: without sources it gives what it gave before, its robust
answers are the reference's tMin rule (the oracle traced from the exact f64 point on the surface), and they survive
moving the origin by eps/4 off or along the surface.  The GPU tests run mfx_bvh_hit_from on three ray families:
(e) closest and any hit from a point on an area-weighted random primitive, (f) any hit toward a point on another primitive (a
light sample's shape) and (g) concave contacts, rays from near an edge toward the primitive across it."""
import ctypes as C
import os

import numpy as np
import pytest

from tests.test_gpu_f32_traversal import (BIG, ORACLE_SCENES, SCENES, _fresh_scene, _gpu_answer, _ptr, _sky,  # noqa: F401
                                          brute, classify, rays)

# which surface-ray queries run: (family, closest or any-hit, tMax); "near" is tMax = (1 - 1e-3) dist, just short of the
# target point, where the frames' own dist - 1e-6 would leave the target pair ambiguous by construction.  (e) as any-hit
# queries are the shadow rays that start into their own sphere (the unlit side near a light's terminator: the chord).
QUERIES = [("e", "closest", BIG), ("e", "any", 2.0), ("f", "any", "near"), ("f", "any", 2.0), ("f", "any", BIG),
           ("g", "closest", BIG)]
CPU_PAIR_BUDGET = 2e7
N_WINDOWS = 64          # the seams take one tMax per call: family (f)'s "near" windows go in groups sorted by dist


def _tmin(desc):
    return 1e-5 if _sky(desc) else 1e-6         # the frames' tMin: ListHit(ray, 0.00001, ..) / Hit(ray, 1e-6, ..)


def _qname(q):
    return f"{q[0]}/{q[1]}/{q[2] if isinstance(q[2], str) else format(q[2], 'g')}"


def classify_from(lib, desc, o, d, src, tmin, tmax, any_hit):
    """classify() for rays that start on primitive src[i] (caller's index, -1 none)."""
    lib.brute_classify_from.restype = C.c_double
    lib.brute_classify_from.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.c_double, C.c_double, C.c_int, C.c_int, C.c_int] + [C.c_void_p] * 7
    o = np.ascontiguousarray(o, np.float64)
    d = np.ascontiguousarray(d, np.float64)
    src = np.ascontiguousarray(src, np.int32)
    n = len(o)
    kind = np.ascontiguousarray(desc.prims["kind"], np.int32)
    v = np.ascontiguousarray(desc.prims["v"], np.float64)
    out = dict(robust=np.zeros(n, np.int8), prim=np.zeros(n, np.int32), sub=np.zeros(n, np.int32), t=np.zeros(n),
               terr=np.zeros(n), eps=np.zeros(n), amb=np.zeros(n, np.int32))
    lib.brute_classify_from(len(kind), _ptr(kind), _ptr(v), n, _ptr(o), _ptr(d), _ptr(src), float(tmin), float(tmax),
                            int(any_hit), int(_sky(desc)), os.cpu_count() or 1, _ptr(out["robust"]), _ptr(out["prim"]),
                            _ptr(out["sub"]), _ptr(out["t"]), _ptr(out["terr"]), _ptr(out["eps"]), _ptr(out["amb"]))
    out["robust"] = out["robust"].astype(bool)
    return out


# ------------------------------------------------------------------ rays that start on a surface
def _f32(p):
    return p.astype(np.float32).astype(np.float64)


def _unit(v):
    return v / np.linalg.norm(v, axis=-1, keepdims=True)


def _tangents(n):
    a = np.where(np.abs(n[:, :1]) < 0.9, np.array([[1.0, 0, 0]]), np.array([[0, 1.0, 0]]))
    t1 = _unit(np.cross(n, a))
    return t1, np.cross(n, t1)


def _subtris(desc):
    """Per primitive: vertices (a, b, c) of its sub-triangles 0 and 1 (a Rect's second half; a copy of the first
    otherwise) and their areas (0 for a missing half, 4 pi r^2 for a sphere)."""
    p = desc.prims
    v = p["v"]
    t0 = np.stack([v[:, 0:3], v[:, 3:6], v[:, 6:9]], 1)
    t1 = np.stack([v[:, 0:3], v[:, 6:9], v[:, 9:12]], 1)
    a0 = 0.5 * np.linalg.norm(np.cross(t0[:, 1] - t0[:, 0], t0[:, 2] - t0[:, 0]), axis=1)
    a1 = np.where(p["kind"] == 1, 0.5 * np.linalg.norm(np.cross(t1[:, 1] - t1[:, 0], t1[:, 2] - t1[:, 0]), axis=1), 0.0)
    sph = p["kind"] == 2
    a0[sph], a1[sph] = 4 * np.pi * v[sph, 3] ** 2, 0.0
    return t0, t1, a0, a1


def surface_points(desc, rng, n, avoid=None):
    """n points in f64 on area-weighted random primitives (a big r >= 32 sphere gets a quarter of the points, not
    nearly all of them), with the primitive, sub-triangle and outward normal.  avoid: per point, a primitive to skip."""
    p = desc.prims
    t0, t1, a0, a1 = _subtris(desc)
    w = a0 + a1
    big = (p["kind"] == 2) & (np.abs(p["v"][:, 3]) >= 32)
    if big.any() and (~big).any():
        w[big] = w[~big].sum() / 3 / big.sum()
    prim = rng.choice(len(p), n, p=w / w.sum())
    if avoid is not None:
        for _ in range(64):
            again = prim == avoid
            if not again.any():
                break
            prim[again] = rng.choice(len(p), int(again.sum()), p=w / w.sum())
        assert not (prim == avoid).any()
    sub = (rng.random(n) * (a0[prim] + a1[prim]) >= a0[prim]).astype(np.int32)
    tri = np.where(sub[:, None, None] == 1, t1[prim], t0[prim])
    bc = rng.random((n, 2))
    flip = bc.sum(1) > 1
    bc[flip] = 1 - bc[flip]
    pts = tri[:, 0] + bc[:, :1] * (tri[:, 1] - tri[:, 0]) + bc[:, 1:] * (tri[:, 2] - tri[:, 0])
    nrm = _unit(np.cross(tri[:, 1] - tri[:, 0], tri[:, 2] - tri[:, 0]))
    sph = p["kind"][prim] == 2
    if sph.any():
        u = _unit(rng.normal(size=(int(sph.sum()), 3)))
        c, r = p["v"][prim[sph], :3], np.abs(p["v"][prim[sph], 3])
        pts[sph], nrm[sph], sub[sph] = c + u * r[:, None], u, 0
    return pts, prim.astype(np.int32), sub, nrm


def _directions(rng, nrm, cos):
    """Unit directions at |cos| to the normals, on a random side, uniform in azimuth."""
    side = np.where(rng.random(len(nrm)) < 0.5, 1.0, -1.0)
    phi = rng.uniform(0, 2 * np.pi, len(nrm))
    t1, t2 = _tangents(nrm)
    s = np.sqrt(np.maximum(0.0, 1 - cos ** 2))
    return _unit((side * cos)[:, None] * nrm + (s * np.cos(phi))[:, None] * t1 + (s * np.sin(phi))[:, None] * t2)


def _eps0(desc, o, prim):
    """The f32 error scale of a point on primitive prim, in the form of the classifier's eps (brute_hit.c header) with
    the primitive's own coordinates where the classifier bounds them by the whole scene's: the shade kernel's hit point
    on it lies that close to the surface, whatever else the scene holds."""
    v, k = desc.prims["v"][prim], desc.prims["kind"][prim]
    sph = k == 2
    coords = np.where(k == 1, np.abs(v[:, :12]).max(1), np.abs(v[:, :9]).max(1))
    coords[sph] = np.abs(v[sph, :3]).max(1) + np.abs(v[sph, 3])
    size = np.where(sph, 2 * np.abs(v[:, 3]),
                    np.linalg.norm(v[:, 3:6] - v[:, :3], axis=1) + np.linalg.norm(v[:, 6:9] - v[:, :3], axis=1))
    return 2.0 ** -24 * (4 * (coords + np.abs(o).max(1)) + 48 * size)


def _shared_edges(desc):
    """(A, sub of A, edge end a, edge end b, apex of A's sub-triangle, B, sub of B) for every edge two primitives share
    exactly, both ways round, where their planes meet at more than 2.5 degrees: the contacts family (g) starts on."""
    p = desc.prims
    v = p["v"]
    edges = {}
    for i, k in enumerate(p["kind"]):
        if k == 2:
            continue
        q = v[i].reshape(4, 3)
        es = [(0, 1, 2, 0), (1, 2, 0, 0), (2, 0, 1, 0)] if k == 0 else [(0, 1, 2, 0), (1, 2, 0, 0), (2, 3, 0, 1), (3, 0, 2, 1)]
        for a, b, c, s in es:
            key = tuple(sorted((q[a].tobytes(), q[b].tobytes())))
            edges.setdefault(key, []).append((i, s, q[a], q[b], q[c]))
    t0, t1, _, _ = _subtris(desc)
    out = []
    with np.errstate(invalid="ignore"):         # a degenerate triangle has no normal and no contact
        for lst in edges.values():
            for A in lst:
                for B in lst:
                    if A[0] == B[0]:
                        continue
                    ta, tb = (t1 if A[1] else t0)[A[0]], (t1 if B[1] else t0)[B[0]]
                    na, nb = _unit(np.cross(ta[1] - ta[0], ta[2] - ta[0])), _unit(np.cross(tb[1] - tb[0], tb[2] - tb[0]))
                    if abs(na @ nb) < np.cos(np.radians(2.5)):
                        out.append((A[0], A[1], A[2], A[3], A[4], B[0], B[1]))
    return out


def has_contacts(desc):
    return len(_shared_edges(desc)) > 0


def surface_rays(desc, family, n, seed=0):
    """(exact f64 origin on the surface, origin rounded to f32, unit direction, source primitive, extra) of a family.
    (e): cosine-distributed on either side of the surface (reflection and transmission) for a third of the rays,
    grazing (|cos| 1e-4 .. 1e-2) for a third, within 5 degrees of the tangent plane for the rest (on spheres: the
    chord and the leaving rays beside it); extra None.  (f): toward a point on another primitive; extra = the distance
    from the f32 origin.  (g): from 10 eps .. 1e-3 (at least 20 eps) off an edge shared with another primitive at an
    angle, toward a point of that primitive; extra None."""
    rng = np.random.default_rng([seed, ord(family)])
    if family in "ef":
        p, src, _sub, nrm = surface_points(desc, rng, n)
        o = _f32(p)
        if family == "e":
            grp = rng.integers(0, 3, n)
            cos = np.where(grp == 0, np.sqrt(rng.random(n)),
                           np.where(grp == 1, 10.0 ** rng.uniform(-4, -2, n), rng.uniform(0, np.sin(np.radians(5)), n)))
            return p, o, _directions(rng, nrm, cos), src, None
        q, _, _, _ = surface_points(desc, rng, n, avoid=src)
        d = q - o
        dist = np.linalg.norm(d, axis=1)
        return p, o, d / dist[:, None], src, dist
    assert family == "g"
    con = _shared_edges(desc)
    pick = rng.integers(0, len(con), n)
    A = np.array([con[k][0] for k in pick], np.int32)
    a, b, c = (np.array([con[k][j] for k in pick]) for j in (2, 3, 4))
    e = a + rng.uniform(0.05, 0.95, (n, 1)) * (b - a)
    h = np.linalg.norm(np.cross(c - a, _unit(b - a)), axis=1)             # height of A's apex over the edge
    eps = _eps0(desc, e, A)
    lo = 10 * eps
    delta = np.minimum(10.0 ** rng.uniform(np.log10(lo), np.log10(np.maximum(1e-3, 20 * lo))), 0.5 * h)
    p = e + (delta / h)[:, None] * (c - e)                                 # on A, delta off the edge
    t0, t1, _, _ = _subtris(desc)
    B, sb = np.array([con[k][5] for k in pick]), np.array([con[k][6] for k in pick])
    tri = np.where(sb[:, None, None] == 1, t1[B], t0[B])
    bc = rng.random((n, 2))
    flip = bc.sum(1) > 1
    bc[flip] = 1 - bc[flip]
    q = tri[:, 0] + bc[:, :1] * (tri[:, 1] - tri[:, 0]) + bc[:, 1:] * (tri[:, 2] - tri[:, 0])
    o = _f32(p)
    return p, o, _unit(q - o), A, None


def kernel_chord(desc, o, d, src):
    """Rays whose source sphere k_f_trace6 re-enters by the chord -2 hb: entering (f32 hb < 0) with an f32 discriminant
    <= 0, computed in numpy as leaf_f3 computes it (a big r >= 32 sphere: big_sphere_roots, in f64 from the f32 ray)
    except that nvcc may fuse a multiply-add, so a ray at the border can fall either way.  Without the chord rule these
    rays would pass through their own sphere."""
    f = np.float32
    v = desc.prims["v"][src]
    sph = (desc.prims["kind"][src] == 2) & (src >= 0)
    big = sph & (np.abs(v[:, 3]) >= 32)
    o32, d32 = o.astype(f), d.astype(f)

    def dot(a, b):
        return (a[:, 0] * b[:, 0] + a[:, 1] * b[:, 1]) + a[:, 2] * b[:, 2]
    oc = o32 - v[:, :3].astype(f)
    hb = dot(oc, d32)
    perp = oc - d32 * hb[:, None]
    small = sph & ~big & (hb < 0) & ((v[:, 3] * v[:, 3]).astype(f) - dot(perp, perp) <= 0)
    ocd = o32.astype(np.float64) - v[:, :3]
    h2 = dot(ocd, d32.astype(np.float64))
    return small | (big & (h2 < 0) & (h2 * h2 - (dot(ocd, ocd) - v[:, 3] ** 2) <= 0))


def _windows(q, dist):
    """(rays, tMax) groups of one query: one group, or for "near" N_WINDOWS groups of rays sorted by distance, each
    with tMax (1 - 1e-3) times its shortest distance -- every target point lies beyond its window."""
    if q[2] != "near":
        return [(np.arange(len(dist)), q[2])]
    order = np.argsort(dist, kind="stable")
    return [(g, (1 - 1e-3) * float(dist[g].min())) for g in np.array_split(order, N_WINDOWS) if len(g)]


def _queries(desc):
    return [q for q in QUERIES if (q[0] != "g" or has_contacts(desc)) and (q[0] != "f" or len(desc.prims) > 1)]


def expected(lib, desc, q, o, d, src, dist):
    """The classifier's answer to query q, window by window, as one set of arrays."""
    out = None
    for g, tmax in _windows(q, dist if dist is not None else np.zeros(len(o))):
        w = classify_from(lib, desc, o[g], d[g], src[g], _tmin(desc), tmax, q[1] == "any")
        if out is None:
            out = {k: np.zeros(len(o), v.dtype) for k, v in w.items()}
        for k in out:
            out[k][g] = w[k]
    return out


def _cpu_rays(name, desc):
    return int(min(SCENES[name][1], max(500, CPU_PAIR_BUDGET / len(desc.prims))))


# Floors on the robust share per scene, in the order of QUERIES (None: not run -- family (g) needs two primitives
# that share an edge at an angle, which the tiny trees, the sphere scenes, the haystack and the two soups of loose
# primitives do not have, and family (f) a second primitive), at 0.8 of the shares measured on the first _cpu_rays()
# rays of each family (DESIGN.md 4.3).  The two haystack runs share one geometry.
FLOORS = {
    "cornell": (0.79, 0.79, 0.79, 0.79, 0.79, 0.33),
    "c1_cube": (0.78, 0.79, 0.79, 0.79, 0.79, 0.30),
    "c2_spot": (0.79, 0.79, 0.79, 0.79, 0.79, 0.41),
    "c3_renault": (0.77, 0.79, 0.80, 0.80, 0.79, 0.48),
    "spheres": (0.79, 0.77, 0.79, 0.79, 0.79, None),
    "haystack_smem12": (0.79, 0.79, 0.79, 0.79, 0.79, None),
    "soup_mixed": (0.78, 0.79, 0.79, 0.79, 0.79, None),
    "soup_km": (0.79, 0.79, 0.79, 0.79, 0.79, None),
    "soup_far_mesh": (0.38, 0.56, 0.73, 0.76, 0.76, 0.52),
    "tiny1": (0.80, 0.80, None, None, None, None),
    "tiny2": (0.80, 0.80, 0.78, 0.79, 0.79, None),
    "tiny3": (0.80, 0.80, 0.80, 0.79, 0.79, None),
    "tiny5": (0.80, 0.80, 0.79, 0.79, 0.79, None),
    "tiny9": (0.80, 0.80, 0.79, 0.79, 0.79, None),
    "sky": (0.79, 0.77, 0.79, 0.79, 0.79, None),
}


def _floor(name, q):
    return FLOORS["haystack_smem12" if name.startswith("haystack") else name][QUERIES.index(q)]


# ------------------------------------------------------------------ CPU: the source rules of the classifier
@pytest.mark.parametrize("name", [s for s in SCENES if s != "haystack_smem1"])
def test_no_source_gives_the_classifier_without_sources(brute, name):
    """src = -1 on every ray gives, array for array, what the classifier without sources gives (families (a)-(c))."""
    desc = SCENES[name][0]()
    n = min(_cpu_rays(name, desc), 4000)
    for fam, kind, tmax in (("a", "closest", BIG), ("a", "any", 0.5), ("b", "closest", BIG), ("c", "any", 2.0)):
        o, d = rays(desc, fam, n)
        want = classify(brute, desc, o, d, 1e-6, tmax, kind == "any")
        got = classify_from(brute, desc, o, d, np.full(n, -1, np.int32), 1e-6, tmax, kind == "any")
        assert all(np.array_equal(got[k], want[k]) for k in want), (fam, kind)


def _non_planar_rects(desc):
    """Rects whose fourth vertex lies off the plane of the first three by more than 1e-12 of their size."""
    v, rect = desc.prims["v"], desc.prims["kind"] == 1
    n = np.cross(v[:, 3:6] - v[:, :3], v[:, 6:9] - v[:, :3])
    off = np.abs(np.einsum("ij,ij->i", n, v[:, 9:12] - v[:, :3]))
    size = np.linalg.norm(n, axis=1) * np.abs(v[:, :12]).max(1)
    return rect & (off > 1e-12 * size)


def _oracle(desc):
    from oracle import oracle
    return oracle.OracleSkyScene(desc) if _sky(desc) else oracle.OracleScene(desc)


def _oracle_hit(orc, desc, o, d):
    """The reference's closest hit from the exact point, tMin as in the frames: (prim, sub, t)."""
    if _sky(desc):
        p, t = orc.hit(o, d, _tmin(desc), BIG)
        return p, np.zeros_like(p), t
    return orc.hit(o, d, _tmin(desc), BIG)


@pytest.mark.parametrize("name", ORACLE_SCENES + ["sky"])
def test_source_rules_are_the_references_tmin_rule(brute, name):
    """The fast path's source rules are the reference's tMin rule done robustly in f32: the oracle, traced from the
    exact f64 point on the surface with the frames' tMin and no source, returns on every robust ray the classifier's
    answer for the f32-rounded point with its source set -- the same primitive and sub-triangle and t within the
    classifier's t error for a closest hit, the same occluded flag for an any-hit query (the oracle's closest hit in
    the window).  These scenes hold no non-planar Rect: the reference would re-hit the other half of one (quirk Q3)
    where the fast path drops both.  Rays with a zero direction component (from one point of an axis-aligned plane to
    another) are left out: the reference's box test divides 0 by 0 there (quirk Q6) and misses boxes the fast path
    enters."""
    desc = SCENES[name][0]()
    assert not _non_planar_rects(desc).any(), f"{name} holds a non-planar Rect: quirk Q3"
    orc = _oracle(desc)
    n = _cpu_rays(name, desc)
    for fam in "efg":
        if not any(q[0] == fam for q in _queries(desc)):
            continue
        p, o, d, src, dist = surface_rays(desc, fam, n)
        keep = (d != 0).all(1)                  # between two points of one axis-aligned plane: quirk Q6
        op, osub, ot = _oracle_hit(orc, desc, p, d)
        for q in (qq for qq in QUERIES if qq[0] == fam):
            want = expected(brute, desc, q, o, d, src, dist)
            r = want["robust"] & keep
            # every case has robust hits, and robust misses unless the rays aim at a primitive inside the window
            assert r.mean() > 0.3 and (want["prim"][r] >= 0).any(), (_qname(q), r.mean())
            assert fam == "g" or q[1] == "any" and q[2] != "near" or (want["prim"][r] < 0).any(), _qname(q)
            if q[1] == "any":
                tmax = np.zeros(n)
                for g, tm in _windows(q, dist if dist is not None else np.zeros(n)):
                    tmax[g] = tm
                bad = r & ((want["prim"] >= 0) != ((op >= 0) & (ot < tmax)))
            else:
                hit = want["prim"] >= 0
                bad = r & ((op != want["prim"]) | (hit & (osub != want["sub"])) | (hit & (np.abs(ot - want["t"]) > want["terr"])))
            assert not bad.any(), f"{name} {_qname(q)}: {int(bad.sum())} robust rays differ from the oracle, first {np.flatnonzero(bad)[:5]}"


@pytest.mark.parametrize("name", ["c1_cube", "c2_spot", "spheres", "soup_far_mesh", "sky"])
def test_source_margins_hold_under_perturbation(brute, name):
    """The shade kernel's f32 hit point can land on either side of the surface.  Robust closest-hit answers of (e) and
    (g) do not change when the origin moves by eps/4 (eps of the source pair) in the tangent plane (the oracle from the
    moved exact point, which stays on the surface) or by eps/4 along the normal to either side (the classifier from the
    moved origin: the reference's tMin rule does not hold off the surface, the source rule does); at most 10 % of the
    robust rays become ambiguous there."""
    desc = SCENES[name][0]()
    assert not _non_planar_rects(desc).any(), f"{name} holds a non-planar Rect: quirk Q3"
    orc = _oracle(desc)
    rng = np.random.default_rng(11)
    v = desc.prims["v"]
    for fam in "eg":
        if fam == "g" and not has_contacts(desc):
            continue
        p, o, d, src, _ = surface_rays(desc, fam, min(_cpu_rays(name, desc), 4000))
        want = classify_from(brute, desc, o, d, src, _tmin(desc), BIG, False)
        r = want["robust"]
        p, o, d, src, wp, ws = p[r], o[r], d[r], src[r], want["prim"][r], want["sub"][r]
        eps = _eps0(desc, o, src)               # the scale of the error of a hit point on the source
        sph = desc.prims["kind"][src] == 2
        t0, t1, _, _ = _subtris(desc)
        nrm = _unit(np.cross(t0[src, 1] - t0[src, 0], t0[src, 2] - t0[src, 0]))
        nrm[sph] = _unit(p[sph] - v[src[sph], :3])
        tan = _unit(np.cross(nrm, _unit(rng.normal(size=nrm.shape))))
        p2 = p + tan * (eps / 4)[:, None]
        p2[sph] = v[src[sph], :3] + _unit(p2[sph] - v[src[sph], :3]) * np.abs(v[src[sph], 3:4])
        op, osub, _ = _oracle_hit(orc, desc, p2, d)
        bad = (op != wp) | ((op >= 0) & (osub != ws))
        assert not bad.any(), f"{name} ({fam}): {int(bad.sum())} robust rays change their answer along the surface"
        for side in (1.0, -1.0):
            got = classify_from(brute, desc, o + side * nrm * (eps / 4)[:, None], d, src, _tmin(desc), BIG, False)
            g = got["robust"]
            bad = g & ((got["prim"] != wp) | ((wp >= 0) & (got["sub"] != ws)))
            assert not bad.any(), f"{name} ({fam}), normal side {side:+}: {int(bad.sum())} robust rays change their answer"
            assert g.mean() >= 0.9, (fam, side, g.mean())


CHORD_SCENES = [s for s in SCENES if s in ("spheres", "sky")]
MIN_CHORD_RAYS = 200


def _robust_chord_rays(want, q, o, d, src, desc):
    """Robust rays of query q whose answer rests on the chord rule: the kernel re-enters the source sphere by the chord,
    and the answer is that sphere (closest hit) or occluded (any hit)."""
    ans = (want["prim"] == src) if q[1] == "closest" else (want["prim"] >= 0)
    return want["robust"] & ans & kernel_chord(desc, o, d, src)


@pytest.mark.parametrize("name", CHORD_SCENES)
def test_chord_rays_are_robust(brute, name):
    """The rays the kernel re-enters their sphere by, near the tangent plane, are robust: hundreds of them per query of
    (e) answer with their own sphere (closest) or occluded (any hit), so dropping the chord rule -- they would then pass
    through their sphere, the terminator incident of DESIGN.md 4.3 -- fails the zero-mismatch test below."""
    desc = SCENES[name][0]()
    _p, o, d, src, _ = surface_rays(desc, "e", _cpu_rays(name, desc))
    chord = kernel_chord(desc, o, d, src)
    for q in (qq for qq in QUERIES if qq[0] == "e"):
        want = classify_from(brute, desc, o, d, src, _tmin(desc), q[2], q[1] == "any")
        k = int(_robust_chord_rays(want, q, o, d, src, desc).sum())
        assert k >= MIN_CHORD_RAYS and k >= 0.9 * chord.sum(), (_qname(q), k, int(chord.sum()))


def _shares(brute, name, n=None):
    desc = SCENES[name][0]()
    n = n or _cpu_rays(name, desc)
    got, fam = {}, {}
    for q in _queries(desc):
        _p, o, d, src, dist = fam.setdefault(q[0], surface_rays(desc, q[0], n))
        got[q] = float(expected(brute, desc, q, o, d, src, dist)["robust"].mean())
    return got


@pytest.mark.parametrize("name", [s for s in SCENES if s != "haystack_smem1"])
def test_surface_robust_shares_meet_their_floors(brute, name):
    """Each case keeps most of its rays robust (a floor at about 0.8 of the measured share), so the zero-mismatch
    tests below cannot pass on an empty set."""
    got = _shares(brute, name)
    assert [f is not None for f in FLOORS[name]] == [q in got for q in QUERIES]
    low = {_qname(q): (got[q], _floor(name, q)) for q in got if got[q] < _floor(name, q)}
    assert not low, low


# ------------------------------------------------------------------ GPU: zero mismatches on robust rays
def _from_answer(s, o, d, src, tmin, q, dist):
    prim, sub, t = np.zeros(len(o), np.int32), np.zeros(len(o), np.int32), np.zeros(len(o))
    for g, tmax in _windows(q, dist if dist is not None else np.zeros(len(o))):
        prim[g], sub[g], t[g] = s.HitFrom(o[g], d[g], src[g], tmin, tmax, any_hit=q[1] == "any")
    return prim, sub, t


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(SCENES))
def test_f32_traversal_from_a_surface_returns_the_f64_answer_on_robust_rays(brute, monkeypatch, tmp_path, name):
    """Every query of families (e)-(g) through mfx_bvh_hit_from: zero mismatches on robust rays (same primitive and
    sub-triangle, t within 1e-5 t + 4 u; the same occluded flag), the robust share at least its floor, and in the
    sphere scenes at least MIN_CHORD_RAYS robust rays of each (e) query whose answer rests on the chord rule."""
    desc = SCENES[name][0]()
    n = SCENES[name][1]
    s = _fresh_scene(monkeypatch, name, desc)
    bad, report, fam = [], [], {}
    for q in _queries(desc):
        _p, o, d, src, dist = fam.setdefault(q[0], surface_rays(desc, q[0], n))
        want = expected(brute, desc, q, o, d, src, dist)
        fp, fsub, ft = _from_answer(s, o, d, src, _tmin(desc), q, dist)
        r = want["robust"]
        if q[1] == "any":
            wrong = r & ((fp >= 0) != (want["prim"] >= 0))
            terr = 0.0
        else:
            hit = want["prim"] >= 0
            wrong = r & ((fp != want["prim"]) | (hit & (fsub != want["sub"])) | (hit & (np.abs(ft - want["t"]) > want["terr"])))
            ok = r & hit & ~wrong
            terr = float((np.abs(ft - want["t"])[ok] / want["t"][ok]).max()) if ok.any() else 0.0
        share = float(r.mean())
        chord = int(_robust_chord_rays(want, q, o, d, src, desc).sum()) if q[0] == "e" else 0
        report.append(f"{_qname(q)}: robust {share:.4f} (floor {_floor(name, q)}), occupied {float((want['prim'][r] >= 0).mean()):.3f}, "
                      f"max rel t error {terr:.2e}, robust chord rays {chord}")
        if name in CHORD_SCENES and q[0] == "e" and chord < MIN_CHORD_RAYS:
            bad.append(f"{_qname(q)}: {chord} robust rays through the chord rule, fewer than {MIN_CHORD_RAYS}")
        if share < _floor(name, q):
            bad.append(f"{_qname(q)}: robust share {share:.4f} under its floor {_floor(name, q)}")
        if wrong.any():
            i = np.flatnonzero(wrong)
            path = tmp_path / f"{name}_{_qname(q).replace('/', '_')}.npz"
            np.savez(path, o=o[i], d=d[i], src=src[i], want_prim=want["prim"][i], want_sub=want["sub"][i],
                     want_t=want["t"][i], got_prim=fp[i], got_sub=fsub[i], got_t=ft[i])
            first = "; ".join(f"o={tuple(o[k])} d={tuple(d[k])} src={src[k]} expected ({want['prim'][k]}, {want['sub'][k]}, "
                              f"{want['t'][k]!r}) got ({fp[k]}, {fsub[k]}, {ft[k]!r})" for k in i[:3])
            bad.append(f"{_qname(q)}: {len(i)} robust rays differ, rays in {path}; first: {first}")
    s.close()
    print(f"\n{name}:\n  " + "\n  ".join(report))
    assert not bad, f"{name}: " + "\n".join(bad)


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(SCENES))
def test_no_source_is_the_fast_seam_bit_for_bit(monkeypatch, name):
    """mfx_bvh_hit_from with src = None returns, bit for bit, what mfx_bvh_hit returns through k_f_trace6
    (MFX_F32_PRIMARY=1 for closest hits, any hit) on the rays of families (a)-(c)."""
    desc = SCENES[name][0]()
    n = min(SCENES[name][1], 20000)
    s = _fresh_scene(monkeypatch, name, desc)
    bad = []
    for fam in "abc":
        o, d = rays(desc, fam, n)
        for q in ((fam, "closest", 1e-6, BIG), (fam, "any", 1e-6, 2.0)):
            want = _gpu_answer(s, monkeypatch, o, d, q)
            got = s.HitFrom(o, d, None, q[2], q[3], any_hit=q[1] == "any")
            if not all(np.array_equal(g, w) for g, w in zip(got, want)):
                bad.append(f"{fam}/{q[1]}")
    s.close()
    assert not bad, f"{name}: differ from mfx_bvh_hit: {bad}"


SUB_BATCHES = (1, 15, 16, 17, 31, 33, 127, 129)


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(SCENES))
def test_surface_answers_do_not_depend_on_the_other_rays(monkeypatch, name):
    """A ray's answer depends on that ray and its source alone, bit for bit: the same rays permuted, sub-batches of 1
    to 129 rays and a fresh scene whose wave holds 1024 paths give the full batch's answers."""
    desc = SCENES[name][0]()
    n = min(SCENES[name][1], 20000)
    fams = [surface_rays(desc, f, n // 2) for f in "ef" if any(q[0] == f for q in _queries(desc))]
    o, d, src = (np.concatenate([f[k] for f in fams]) for k in (1, 2, 3))
    perm = np.random.default_rng(5).permutation(len(o))
    tmin = _tmin(desc)
    queries = [(False, BIG), (True, 2.0)]
    s = _fresh_scene(monkeypatch, name, desc)
    want = {q: s.HitFrom(o, d, src, tmin, q[1], any_hit=q[0]) for q in queries}
    bad = []
    for q in queries:
        got = s.HitFrom(o[perm], d[perm], src[perm], tmin, q[1], any_hit=q[0])
        if not all(np.array_equal(g, w[perm]) for g, w in zip(got, want[q])):
            bad.append(f"any={q[0]}: permuted rays")
        for k in SUB_BATCHES:
            got = s.HitFrom(o[:k], d[:k], src[:k], tmin, q[1], any_hit=q[0])
            if not all(np.array_equal(g, w[:k]) for g, w in zip(got, want[q])):
                bad.append(f"any={q[0]}: a batch of the first {k} rays")
    s.close()
    s = _fresh_scene(monkeypatch, name, desc, MFX_WAVE_PATHS="1024")
    for q in queries:
        got = s.HitFrom(o, d, src, tmin, q[1], any_hit=q[0])
        if not all(np.array_equal(g, w) for g, w in zip(got, want[q])):
            bad.append(f"any={q[0]}: MFX_WAVE_PATHS=1024")
    s.close()
    assert not bad, f"{name}: answers change with " + ", ".join(bad)


@pytest.mark.gpu
def test_source_outside_the_scene_is_rejected(monkeypatch):
    """A source index outside [-1, n_prims) is an error before anything runs on the device, not a ray without one."""
    from mafrixraytracing_b200 import _lib
    desc = SCENES["tiny3"][0]()
    s = _fresh_scene(monkeypatch, "tiny3", desc)
    o, d = np.zeros((2, 3)), np.tile([0.0, 0.0, -1.0], (2, 1))
    for bad in (-2, len(desc.prims)):
        with pytest.raises(_lib.MafrixError, match="outside"):
            s.HitFrom(o, d, [0, bad], 1e-6, BIG)
    assert s.HitFrom(o, d, [len(desc.prims) - 1, -1], 1e-6, BIG)[0].shape == (2,)
    s.close()
