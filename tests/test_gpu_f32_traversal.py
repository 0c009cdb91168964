"""The f32 traversal (k_f_trace6) query by query against a brute-force f64 reference, with no tolerance on the rays
whose answer does not depend on rounding.

tests/native/brute_hit.c tests every ray against every primitive in f64 with the fast path's stated semantics
(DESIGN.md 4.3) and classifies each (ray, primitive) pair as a clear hit, a clear miss or ambiguous at margins derived
from the f32 kernel's error (its header states them).  A ray whose answer is the same however its ambiguous pairs are
resolved is ROBUST, and on robust rays the kernel must return the f64 answer: the same primitive and sub-triangle and
t within 1e-5 relative plus the t margin for a closest hit, the same occluded flag for an any-hit query.  The CPU tests
check the classifier itself first: its robust answers are the oracle's, they survive perturbations of the ray below
the margins, and each case keeps a floor on its robust share so that no test can pass on an empty set.

The closest-hit seam runs k_f_trace6 with MFX_F32_PRIMARY=1 (otherwise it takes the id-exact kernel), the any-hit
seam runs k_f_trace6<ANY>; the sphere scenes hold an r = 1000 sphere, so they run the BIG instances."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from mafrixraytracing_b200 import scenes
from mafrixraytracing_b200.scene import (PATH_INTEGRATOR, AreaLight, PinholeCamera, SceneDesc, make_materials)
from tests.conftest import ROOT
from tests.test_gpu_hybrid_stress import _soup
from tests.test_gpu_parity import tiny_tree_scene
from tests.test_gpu_traversal_stack import _haystack

BIG = 99999999.
TMIN = 1e-6


# ------------------------------------------------------------------ the classifier
@pytest.fixture(scope="module")
def brute(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("brute") / "libbrute_hit.so")
    subprocess.check_call(["/usr/bin/gcc", "-O2", "-shared", "-fPIC", "-pthread", "-o", so,
                           os.path.join(ROOT, "tests", "native", "brute_hit.c"), "-lm"])
    lib = C.CDLL(so)
    P = C.c_void_p
    lib.brute_classify.restype = C.c_double
    lib.brute_classify.argtypes = [C.c_int, P, P, C.c_int, P, P, C.c_double, C.c_double, C.c_int, C.c_int, C.c_int,
                                   P, P, P, P, P, P, P]
    return lib


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def classify(lib, desc, o, d, tmin, tmax, any_hit):
    """Per ray: robust flag, expected (prim, sub, t) -- prim >= 0 is 'occluded' for an any-hit query -- the allowed t
    error of a robust closest hit, the margin eps of its winning pair and the number of ambiguous pairs."""
    o = np.ascontiguousarray(o, np.float64)
    d = np.ascontiguousarray(d, np.float64)
    n = len(o)
    kind = np.ascontiguousarray(desc.prims["kind"], np.int32)
    v = np.ascontiguousarray(desc.prims["v"], np.float64)
    out = dict(robust=np.zeros(n, np.int8), prim=np.zeros(n, np.int32), sub=np.zeros(n, np.int32), t=np.zeros(n),
               terr=np.zeros(n), eps=np.zeros(n), amb=np.zeros(n, np.int32))
    lib.brute_classify(len(kind), _ptr(kind), _ptr(v), n, _ptr(o), _ptr(d), float(tmin), float(tmax), int(any_hit),
                       int(_sky(desc)), os.cpu_count() or 1, _ptr(out["robust"]), _ptr(out["prim"]), _ptr(out["sub"]),
                       _ptr(out["t"]), _ptr(out["terr"]), _ptr(out["eps"]), _ptr(out["amb"]))
    out["robust"] = out["robust"].astype(bool)
    return out


# ------------------------------------------------------------------ scenes
def _soup_desc(seed, n_tri, n_rect, n_sph, scale, offset, grid):
    """One scene of test_gpu_hybrid_stress: its primitives, a light and a camera of the same scale."""
    offset = np.array(offset, float)
    prims = _soup(np.random.default_rng(seed), n_tri, n_rect, n_sph, scale, offset, grid)
    light = AreaLight(np.array([(-1, 3, 1), (-1, 3, -1), (1, 3, -1), (1, 3, 1)], float) * scale + offset, (0, -1, 0), (10, 10, 10))
    cam = PinholeCamera(offset + np.array([0.3, 0.8, 3.5]) * scale, (-0.05, -0.2, -1), 120.0, 1.0)
    return SceneDesc(prims, make_materials([("lambert", (0.7, 0.7, 0.7))]), light, cam, 64, 64, 2, PATH_INTEGRATOR)


# name: (builder, rays per family, environment of the GPU run).  Rays per family are fewer where the brute force costs
# more (C3: 37 k primitives).
SCENES = {
    "cornell": (lambda: scenes.cornell(width=8, height=8), 100000, {}),
    "c1_cube": (lambda: scenes.c1_cube(width=8, height=8), 100000, {}),
    "c2_spot": (lambda: scenes.c2_spot(width=8, height=8), 40000, {}),
    "c3_renault": (lambda: scenes.c3_renault(width=8, height=8), 6000, {}),
    "spheres": (lambda: scenes.c4_spheres(width=8, height=8, grid=30), 100000, {}),
    "haystack_smem12": (lambda: _haystack(width=16, height=9), 40000, {"MFX_STACK_SMEM": "12"}),
    "haystack_smem1": (lambda: _haystack(width=16, height=9), 40000, {"MFX_STACK_SMEM": "1"}),
    "soup_mixed": (lambda: _soup_desc(1, 400, 20, 20, 1.0, (0, 0, 0), False), 100000, {}),
    "soup_km": (lambda: _soup_desc(4, 500, 30, 10, 1e3, (0, 0, 0), False), 100000, {}),
    "soup_far_mesh": (lambda: _soup_desc(6, 2000, 0, 0, 0.01, (100.0, 100.0, 100.0), True), 100000, {}),
    **{f"tiny{k}": ((lambda k=k: tiny_tree_scene(k)), 100000, {}) for k in (1, 2, 3, 5, 9)},
    "sky": (lambda: scenes.random_scene(width=8, height=4), 100000, {}),
}


def _sky(desc):
    return desc.sky is not None


def _has_spheres(desc):
    return bool((desc.prims["kind"] == 2).any())


def _box(desc):
    """Bounds of the scene without its big (r >= 32) spheres: rays start around the geometry, not around a planet."""
    p = desc.prims
    lo, hi = np.full(3, np.inf), np.full(3, -np.inf)
    for k, row in zip(p["kind"], p["v"]):
        if k == 2:
            if abs(row[3]) >= 32:
                continue
            lo, hi = np.minimum(lo, row[:3] - abs(row[3])), np.maximum(hi, row[:3] + abs(row[3]))
        else:
            pts = row[:12 if k == 1 else 9].reshape(-1, 3)
            lo, hi = np.minimum(lo, pts.min(0)), np.maximum(hi, pts.max(0))
    return lo, hi


def _unit(rng, n):
    d = rng.normal(size=(n, 3))
    return d / np.linalg.norm(d, axis=1)[:, None]


def _points_on_prims(desc, rng, n):
    p = desc.prims[rng.integers(0, len(desc.prims), n)]
    out = np.empty((n, 3))
    w = rng.random((n, 2))
    flip = w.sum(1) > 1
    w[flip] = 1 - w[flip]
    for i, (k, v) in enumerate(zip(p["kind"], p["v"])):
        if k == 2:
            out[i] = v[:3] + _unit(rng, 1)[0] * abs(v[3]) * rng.random() ** (1 / 3)
        else:
            s = int(rng.integers(0, 2)) if k == 1 else 0
            a, b, c = v[0:3], v[3 * (1 + s):3 * (2 + s)], v[3 * (2 + s):3 * (3 + s)]
            out[i] = a + w[i, 0] * (b - a) + w[i, 1] * (c - a)
    return out


def rays(desc, family, n, seed=0):
    """(o, d) of one ray family: (a) origins in the scene box enlarged 1.5x, unit directions; (b) from outside the box,
    aimed at random points of random primitives; (c) axis-parallel: one or two components 0.0 or -0.0; (d) (a) with
    |d| from 1e-3 to 1e3 (triangle scenes only: Sphere.Hit takes a unit direction)."""
    rng = np.random.default_rng([seed, ord(family)])
    lo, hi = _box(desc)
    c, h = 0.5 * (lo + hi), 0.5 * (hi - lo)
    if family in "ad":
        o = c + h * 1.5 * rng.uniform(-1, 1, (n, 3))
        d = _unit(rng, n)
        if family == "d":
            d *= 10.0 ** rng.uniform(-3, 3, (n, 1))
    elif family == "b":
        u = _unit(rng, n)
        if _has_spheres(desc):
            u[:, 1] = np.abs(u[:, 1])                     # above the ground sphere
        o = c + u * (1.5 * np.linalg.norm(h) + 1e-3)
        d = _points_on_prims(desc, rng, n) - o
        d /= np.linalg.norm(d, axis=1)[:, None]
    else:
        o = c + h * 1.5 * rng.uniform(-1, 1, (n, 3))
        d = _unit(rng, n)
        zero = rng.random((n, 3)) < np.where(rng.random((n, 1)) < 0.5, 1 / 3, 2 / 3)
        zero[zero.all(1), rng.integers(0, 3)] = False
        zero[~zero.any(1), 0] = True
        d[zero] = np.where(rng.random(zero.sum()) < 0.5, 0.0, -0.0)
        d /= np.linalg.norm(d, axis=1)[:, None]
    return o, d


# (family, closest or any-hit, tMin, tMax): (e) is family (a) with tMin 0.25, (f) family (a) with four shadow windows
QUERIES = [("a", "closest", TMIN, BIG), ("a", "any", TMIN, 0.05), ("a", "any", TMIN, 0.5), ("a", "any", TMIN, 2.0),
           ("a", "any", TMIN, BIG), ("b", "closest", TMIN, BIG), ("b", "any", TMIN, 2.0), ("c", "closest", TMIN, BIG),
           ("c", "any", TMIN, 2.0), ("d", "closest", TMIN, BIG), ("d", "any", TMIN, 2.0), ("a", "closest", 0.25, BIG),
           ("a", "closest", 0.25, 1.0)]


def _queries(desc):
    return [q for q in QUERIES if not (q[0] == "d" and _has_spheres(desc))]


def _qname(q):
    fam, kind, tmin, tmax = q
    return f"{fam}/{kind}/{tmin:g}/{tmax:g}"


# Floors on the robust share per scene, in the order of QUERIES (None: not run), at about 0.8 of the shares measured on
# the first _cpu_rays() rays of each family (DESIGN.md 4.3).  The two haystack runs share one geometry.
FLOORS = {
    "cornell": (0.79, 0.80, 0.79, 0.80, 0.80, 0.79, 0.79, 0.80, 0.80, 0.79, 0.79, 0.79, 0.79),
    "c1_cube": (0.79, 0.80, 0.79, 0.79, 0.79, 0.79, 0.80, 0.80, 0.80, 0.79, 0.79, 0.79, 0.80),
    "c2_spot": (0.79, 0.80, 0.80, 0.79, 0.79, 0.79, 0.80, 0.80, 0.80, 0.80, 0.80, 0.79, 0.80),
    "c3_renault": (0.80, 0.80, 0.80, 0.80, 0.80, 0.77, 0.80, 0.79, 0.80, 0.80, 0.80, 0.80, 0.80),
    "spheres": (0.79, 0.78, 0.78, 0.78, 0.79, 0.79, 0.79, 0.78, 0.78, None, None, 0.78, 0.78),
    "haystack_smem12": (0.79, 0.80, 0.79, 0.79, 0.79, 0.77, 0.80, 0.79, 0.80, 0.79, 0.79, 0.79, 0.79),
    "soup_mixed": (0.79, 0.80, 0.80, 0.80, 0.80, 0.79, 0.79, 0.79, 0.80, None, None, 0.79, 0.79),
    "soup_km": (0.79, 0.80, 0.80, 0.80, 0.79, 0.79, 0.80, 0.79, 0.80, None, None, 0.79, 0.80),
    "soup_far_mesh": (0.67, 0.73, 0.73, 0.73, 0.73, 0.38, 0.66, 0.71, 0.75, 0.69, 0.74, 0.80, 0.80),
    "tiny1": (0.80, 0.80, 0.80, 0.80, 0.80, 0.79, 0.79, 0.80, 0.80, 0.79, 0.80, 0.80, 0.80),
    "tiny2": (0.80, 0.80, 0.80, 0.80, 0.80, 0.79, 0.79, 0.80, 0.80, 0.80, 0.80, 0.80, 0.80),
    "tiny3": (0.80, 0.80, 0.80, 0.80, 0.80, 0.79, 0.79, 0.80, 0.80, 0.80, 0.80, 0.80, 0.80),
    "tiny5": (0.80, 0.80, 0.80, 0.80, 0.80, 0.79, 0.79, 0.80, 0.80, 0.80, 0.80, 0.80, 0.80),
    "tiny9": (0.80, 0.80, 0.80, 0.80, 0.80, 0.79, 0.79, 0.80, 0.80, 0.80, 0.80, 0.80, 0.80),
    "sky": (0.79, 0.79, 0.79, 0.79, 0.79, 0.79, 0.79, 0.79, 0.79, None, None, 0.79, 0.79),
}
CPU_PAIR_BUDGET = 2e7


def _floor(name, q):
    return FLOORS["haystack_smem12" if name.startswith("haystack") else name][QUERIES.index(q)]


def _cpu_rays(name, desc):
    return int(min(SCENES[name][1], max(500, CPU_PAIR_BUDGET / len(desc.prims))))


# ------------------------------------------------------------------ CPU: the reference before the GPU is held to it
ORACLE_SCENES = ["c1_cube", "c2_spot", "c3_renault", "spheres", "haystack_smem12", "soup_far_mesh", "tiny9"]


@pytest.mark.parametrize("name", ORACLE_SCENES)
def test_classifier_agrees_with_the_oracle(brute, name):
    """On robust closest-hit rays the oracle (the reference's semantics, its own tree) returns the classifier's
    primitive, sub-triangle and t to 1e-12.  These scenes hold no non-planar Rect, where quirks Q2 and Q3 could make
    the reference differ from the fast semantics (Cornell's left wall is one).  Family (c) is left out: with a zero
    direction component the reference's box test divides 0 by 0 (quirk Q6) and misses boxes the fast path enters."""
    from oracle import oracle
    desc = SCENES[name][0]()
    orc = oracle.OracleScene(desc)
    n = _cpu_rays(name, desc)
    for fam in ("a", "b") + (() if _has_spheres(desc) else ("d",)):
        o, d = rays(desc, fam, n)
        want = classify(brute, desc, o, d, TMIN, BIG, False)
        op, osub, ot = orc.hit(o, d, TMIN, BIG)
        r = want["robust"]
        assert r.mean() > 0.3 and (want["prim"][r] >= 0).any(), (fam, r.mean())
        bad = r & ((op != want["prim"]) | ((op >= 0) & (osub != want["sub"])) |
                   ((op >= 0) & (np.abs(ot - want["t"]) > 1e-12 * np.abs(want["t"]))))
        assert not bad.any(), f"{name} family {fam}: {int(bad.sum())} robust rays differ from the oracle, first {np.flatnonzero(bad)[:5]}"


@pytest.mark.parametrize("name", ["c1_cube", "c2_spot", "spheres", "haystack_smem12", "soup_far_mesh"])
def test_margins_hold_under_perturbation(brute, name):
    """Each robust closest-hit ray moved 4 times in f64 -- o by up to eps/4 in a random direction, d by the same
    relative amount -- must keep the oracle's answer: the margins hold on the real geometry."""
    from oracle import oracle
    desc = SCENES[name][0]()
    orc = oracle.OracleScene(desc)
    rng = np.random.default_rng(7)
    for fam in ("a", "b"):
        o, d = rays(desc, fam, min(_cpu_rays(name, desc), 4000))
        want = classify(brute, desc, o, d, TMIN, BIG, False)
        r = want["robust"]
        o, d, wp, ws, eps = o[r], d[r], want["prim"][r], want["sub"][r], want["eps"][r]
        rel = eps / (np.abs(o).max(1) + np.abs(desc.prims["v"]).max())        # eps over its largest length
        for _ in range(4):
            o2 = o + _unit(rng, len(o)) * (eps / 4 * rng.random(len(o)))[:, None]
            d2 = d + _unit(rng, len(d)) * (np.linalg.norm(d, axis=1) * rel / 4 * rng.random(len(d)))[:, None]
            op, osub, _ = orc.hit(o2, d2, TMIN, BIG)
            bad = (op != wp) | ((op >= 0) & (osub != ws))
            assert not bad.any(), f"{name} family {fam}: {int(bad.sum())} perturbed robust rays change their answer"


def _shares(brute, name, n=None):
    desc = SCENES[name][0]()
    n = n or _cpu_rays(name, desc)
    got, fam = {}, {}
    for q in _queries(desc):
        o, d = fam.setdefault(q[0], rays(desc, q[0], n))
        got[q] = float(classify(brute, desc, o, d, q[2], q[3], q[1] == "any")["robust"].mean())
    return got


@pytest.mark.parametrize("name", [s for s in SCENES if s != "haystack_smem1"])
def test_robust_shares_meet_their_floors(brute, name):
    """Each case keeps most of its rays robust (a floor at about 0.8 of the measured share), so the zero-mismatch
    tests below cannot pass on an empty set."""
    got = _shares(brute, name)
    assert [f is not None for f in FLOORS[name]] == [q in got for q in QUERIES]
    low = {_qname(q): (got[q], _floor(name, q)) for q in got if got[q] < _floor(name, q)}
    assert not low, low


# ------------------------------------------------------------------ GPU: zero mismatches on robust rays
def _gpu_answer(s, monkeypatch, o, d, q):
    from mafrixraytracing_b200 import FAST_F32
    _fam, kind, tmin, tmax = q
    if kind == "any":
        return s.Hit(o, d, tmin, tmax, precision=FAST_F32, any_hit=True)
    monkeypatch.setenv("MFX_F32_PRIMARY", "1")          # k_f_trace6, not the id-exact kernel
    try:
        return s.Hit(o, d, tmin, tmax, precision=FAST_F32)
    finally:
        monkeypatch.delenv("MFX_F32_PRIMARY")


def _fresh_scene(monkeypatch, name, desc, **env):
    from mafrixraytracing_b200 import Scene
    for k, v in {**SCENES[name][2], **env}.items():
        monkeypatch.setenv(k, v)
    return Scene(desc)


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(SCENES))
def test_f32_traversal_returns_the_f64_answer_on_robust_rays(brute, monkeypatch, tmp_path, name):
    """Every query of every ray family: zero mismatches on robust rays (same primitive and sub-triangle, t within
    1e-5 t + 4 u; the same occluded flag), and the robust share at least its floor."""
    desc = SCENES[name][0]()
    n = SCENES[name][1]
    s = _fresh_scene(monkeypatch, name, desc)
    bad, report = [], []
    fam = {}
    for q in _queries(desc):
        o, d = fam.setdefault(q[0], rays(desc, q[0], n))
        want = classify(brute, desc, o, d, q[2], q[3], q[1] == "any")
        fp, fsub, ft = _gpu_answer(s, monkeypatch, o, d, q)
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
        report.append(f"{_qname(q)}: robust {share:.4f} (floor {_floor(name, q)}), occupied {float((want['prim'][r] >= 0).mean()):.3f}, "
                      f"max rel t error {terr:.2e}")
        if share < _floor(name, q):
            bad.append(f"{_qname(q)}: robust share {share:.4f} under its floor {_floor(name, q)}")
        if wrong.any():
            i = np.flatnonzero(wrong)
            path = tmp_path / f"{name}_{_qname(q).replace('/', '_')}.npz"
            np.savez(path, o=o[i], d=d[i], tmin=q[2], tmax=q[3], want_prim=want["prim"][i], want_sub=want["sub"][i],
                     want_t=want["t"][i], got_prim=fp[i], got_sub=fsub[i], got_t=ft[i])
            first = "; ".join(f"o={tuple(o[k])} d={tuple(d[k])} expected ({want['prim'][k]}, {want['sub'][k]}, {want['t'][k]!r}) "
                              f"got ({fp[k]}, {fsub[k]}, {ft[k]!r})" for k in i[:3])
            bad.append(f"{_qname(q)} (tMin {q[2]}, tMax {q[3]}): {len(i)} robust rays differ, rays in {path}; first: {first}")
    s.close()
    print(f"\n{name}:\n  " + "\n  ".join(report))
    assert not bad, f"{name}: " + "\n".join(bad)


SUB_BATCHES = (1, 15, 16, 17, 31, 33, 127, 129)


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(SCENES))
def test_f32_answers_do_not_depend_on_the_other_rays(monkeypatch, name):
    """A ray's answer depends on that ray alone, robust or not, bit for bit: the same rays permuted, a fresh scene
    whose wave holds 1024 paths (the seam's chunk loop over many chunks) and sub-batches around the refill threshold
    (16) and the warp and block sizes give the full batch's answers."""
    desc = SCENES[name][0]()
    n = min(SCENES[name][1], 20000)
    o, d = np.concatenate([rays(desc, f, n // 2)[0] for f in "bc"]), np.concatenate([rays(desc, f, n // 2)[1] for f in "bc"])
    perm = np.random.default_rng(5).permutation(len(o))
    queries = [("b", "closest", TMIN, BIG), ("b", "any", TMIN, 2.0)]
    s = _fresh_scene(monkeypatch, name, desc)
    want = {q: _gpu_answer(s, monkeypatch, o, d, q) for q in queries}
    bad = []
    for q in queries:
        got = _gpu_answer(s, monkeypatch, o[perm], d[perm], q)
        if not all(np.array_equal(g, w[perm]) for g, w in zip(got, want[q])):
            bad.append(f"{q[1]}: permuted rays")
        for k in SUB_BATCHES:
            got = _gpu_answer(s, monkeypatch, o[:k], d[:k], q)
            if not all(np.array_equal(g, w[:k]) for g, w in zip(got, want[q])):
                bad.append(f"{q[1]}: a batch of the first {k} rays")
    s.close()
    s = _fresh_scene(monkeypatch, name, desc, MFX_WAVE_PATHS="1024")
    for q in queries:
        got = _gpu_answer(s, monkeypatch, o, d, q)
        if not all(np.array_equal(g, w) for g, w in zip(got, want[q])):
            bad.append(f"{q[1]}: MFX_WAVE_PATHS=1024")
    s.close()
    assert not bad, f"{name}: answers change with " + ", ".join(bad)
