"""The own-tree traversal stack and its spill columns.

The own-tree kernels (k_f_trace6, <TAIL> included, and the id-exact k_h_trace) keep the
first MFX_STACK_SMEM deferred-hit entries of a lane (default 12) in shared memory and everything deeper in a per-thread
column of a global buffer, sized for 3*depth entries, the most a walk of the tree can push.  Where a value lives must
not change an answer: every query and every frame below is compared bit for bit across shared-memory budgets of 1, 2
and 3 entries (a 3-entry push straddles the boundary), the shipped 12 and one that holds the whole stack, and in frames
across one and two streams: the two-stream mode runs the shadow queries of bounce b beside the closest hits of bounce
b+1, and each of the two launches must have spill columns of its own.

The haystack (thin straws in a cube) is the scene that makes the stack deep: the CPU model of the traversal
(tools/own_tree_sim.cpp) shows that most of its rays go beyond 12 entries, which is what makes the GPU tests here
exercise the spill columns at the shipped setting."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from mafrixraytracing_b200 import scenes
from mafrixraytracing_b200.scene import (PATH_INTEGRATOR, AreaLight, PinholeCamera, SceneDesc, make_materials, make_prims)
from tests.conftest import ROOT

BIG = 99999999.
ALL_SHARED = "48"       # the largest budget that fits 48 KB of shared memory at 128 threads: the haystack needs 27 entries


def _haystack(n=5000, length=1.5, seed=1, integrator=PATH_INTEGRATOR, width=160, height=90, max_depth=5):
    """n thin triangles ("straws") of the given length with random centres in [-1,1]^3 and random directions, over a
    floor, lit by a 1x1 quad above.  Their boxes overlap everywhere, so a ray keeps many deferred subtrees."""
    rng = np.random.default_rng(seed)
    c = rng.uniform(-1, 1, (n, 3))
    d = rng.normal(size=(n, 3))
    d /= np.linalg.norm(d, axis=1)[:, None]
    w = np.cross(d, rng.normal(size=(n, 3)))
    w /= np.linalg.norm(w, axis=1)[:, None]
    straws = make_prims(n)
    straws["v"][:, 0:3] = c - 0.5 * length * d
    straws["v"][:, 3:6] = c + 0.5 * length * d
    straws["v"][:, 6:9] = c + 0.01 * w
    floor = scenes.quad_facing((-4, -1.5, -4), (-4, -1.5, 4), (4, -1.5, 4), (4, -1.5, -4), (0, 1, 0), 0)
    mats = make_materials([("lambert", scenes.WHITE)])
    light = AreaLight(np.array([(-0.5, 2.5, 0.5), (-0.5, 2.5, -0.5), (0.5, 2.5, -0.5), (0.5, 2.5, 0.5)], float), (0, -1, 0), (10, 10, 10))
    cam = PinholeCamera((0, 0.2, -4), (0, 0, 1), 120.0, 16.0 / 9.0)
    return SceneDesc(np.concatenate([straws, floor]), mats, light, cam, width, height, max_depth, integrator, name="haystack")


def _desc(name, **kw):
    if name == "haystack":
        return _haystack(**kw)
    if name == "spheres":
        return scenes.c4_spheres(grid=30, **kw)
    return scenes.WORKLOADS[name](**kw)


# ------------------------------------------------------------------ CPU model: how deep the stack goes
def _stack_model(tmp_path, desc, width, height):
    exe = str(tmp_path / "own_tree_sim")
    csrc = os.path.join(ROOT, "mafrixraytracing_b200", "csrc")
    if not os.path.exists(exe):
        subprocess.check_call(["/usr/bin/g++", "-std=c++17", "-O2", "-pthread", "-I", "/usr/local/cuda/include", "-I", csrc, "-o", exe,
                               os.path.join(ROOT, "tools", "own_tree_sim.cpp"), os.path.join(csrc, "mfx_build.cpp")])
    tris = []
    for p in desc.prims:
        tris.append(p["v"][:9])
        if p["kind"] == 1:                                    # a Rect is two triangles, as the fast path slots it
            tris.append(np.concatenate([p["v"][0:3], p["v"][6:9], p["v"][9:12]]))
    path = str(tmp_path / f"{desc.name}.bin")
    np.array(tris, np.float64).tofile(path)
    cam, lp = desc.camera, desc.light.p
    view = [*cam.pos_arg, *cam.dir_arg, cam.fov, cam.aspect, *lp[0], *lp[1], *lp[3], min(desc.max_depth, 5)]
    out = subprocess.check_output([exe, path, str(len(tris)), str(width), str(height)] + [repr(float(x)) for x in view], text=True,
                                  env={k: v for k, v in os.environ.items() if k != "MFX_STACK_SMEM"})
    got = {}
    for kind, peak, bound, deep, rays, smem in re.findall(r"stack, (\w+): peak (\d+) entries, 3\*depth (\d+); (\d+) of (\d+) rays above (\d+) entries", out):
        assert int(smem) == 12
        got[kind] = dict(peak=int(peak), bound=int(bound), deep=int(deep) / int(rays))
    assert set(got) == {"closest", "shadow"}, out
    return got


def test_stack_bound_holds_and_the_haystack_spills_in_the_cpu_model(tmp_path):
    """The spill columns hold 3*depth - MFX_STACK_SMEM entries per thread: no query of the model may push deeper than
    3*depth.  On the haystack most rays must go beyond the 12 shared entries of the shipped kernels, so that the GPU
    tests below run the global half of the stack on most of their rays, not on a few."""
    hay = _stack_model(tmp_path, _haystack(), 160, 90)
    c3 = _stack_model(tmp_path, scenes.c3_renault(), 96, 54)
    for got in (hay, c3):
        for q in got.values():
            assert 0 < q["peak"] <= q["bound"], got
    assert hay["closest"]["bound"] > 12 and c3["closest"]["bound"] > 48       # both trees have spill columns; C3's even at the clamp
    assert hay["closest"]["deep"] >= 0.30 and hay["shadow"]["deep"] >= 0.20, hay


# ------------------------------------------------------------------ GPU: where an entry lives changes no answer
def _fast_bytes(monkeypatch, desc, smem):
    from mafrixraytracing_b200 import Scene
    monkeypatch.setenv("MFX_STACK_SMEM", smem)
    s = Scene(desc)
    b = s.device_bytes()["fast"]
    s.close()
    return b


@pytest.mark.gpu
@pytest.mark.parametrize("name,kw", [("haystack", dict(width=16, height=9)), ("c3_renault", dict(width=8, height=8)),
                                     ("spheres", dict(width=8, height=8))])
def test_seams_do_not_depend_on_the_shared_stack_budget(monkeypatch, name, kw):
    """Bvh.Hit through the production kernels with 1, 2, 3, 12 and all stack entries in shared memory (the knob is read
    when a scene's layout is built: a fresh scene per value).  The id-exact closest hits (k_h_trace) must be the
    oracle's ids, sub-triangles and t every time; the f32 closest hits (k_f_trace6) and the any-hit answers at two tMax
    must be the all-in-shared run's, bit for bit.  The sphere scene also runs the kernels' f64 big-sphere branch."""
    from mafrixraytracing_b200 import Scene, FAST_F32
    from oracle import oracle
    desc = _desc(name, **kw)
    rng = np.random.default_rng(3)
    n = 100000
    org = rng.uniform(-3, 3, (n, 3))
    if name == "spheres":
        org[:, 1] = rng.uniform(0.05, 3, n)
    d = rng.normal(size=(n, 3))
    d /= np.linalg.norm(d, axis=1)[:, None]
    op, osub, ot = oracle.OracleScene(desc).hit(org, d, 1e-6, BIG)
    assert (op >= 0).mean() > 0.2
    got = {}
    monkeypatch.delenv("MFX_F32_PRIMARY", raising=False)
    for smem in (ALL_SHARED, "12", "3", "2", "1"):
        monkeypatch.setenv("MFX_STACK_SMEM", smem)
        s = Scene(desc)
        fp, fsub, ft = s.Hit(org, d, 1e-6, BIG, precision=FAST_F32)
        assert np.array_equal(fp, op) and np.array_equal(fsub, osub) and np.array_equal(ft, ot), smem
        monkeypatch.setenv("MFX_F32_PRIMARY", "1")
        f32 = s.Hit(org, d, 1e-6, BIG, precision=FAST_F32)
        monkeypatch.delenv("MFX_F32_PRIMARY")
        anyhit = [s.Hit(org, d, 1e-6, tmax, precision=FAST_F32, any_hit=True)[0] for tmax in (0.5, 2.0)]
        got[smem] = (f32, anyhit)
        s.close()
    f32_0, any_0 = got[ALL_SHARED]
    assert (f32_0[0] >= 0).any() and all((a >= 0).any() and (a < 0).any() for a in any_0)
    for smem, (f32, anyhit) in got.items():
        assert all(np.array_equal(a, b) for a, b in zip(f32, f32_0)), f"f32 closest hits differ at MFX_STACK_SMEM={smem}"
        for tmax, a, b in zip((0.5, 2.0), anyhit, any_0):
            assert np.array_equal(a, b), f"any-hit answers at tMax {tmax} differ at MFX_STACK_SMEM={smem}"
    assert _fast_bytes(monkeypatch, desc, "1") > _fast_bytes(monkeypatch, desc, ALL_SHARED)      # the small budgets did spill


def _frame(monkeypatch, desc, spp, seed=3, smem=None, two=None):
    """One fast Sample on a fresh scene under the given knobs: (frame, closest rays, shadow rays)."""
    from mafrixraytracing_b200 import Scene, CudaPixelIntegrator, FAST_F32
    for var, val in (("MFX_STACK_SMEM", smem), ("MFX_TWO_STREAMS", two)):
        if val is None:
            monkeypatch.delenv(var, raising=False)
        else:
            monkeypatch.setenv(var, val)
    s = Scene(desc)
    integ = CudaPixelIntegrator(s, precision=FAST_F32, seed=seed)
    img = integ.Sample(spp).copy()
    st = integ.stats
    s.close()
    return img, st["closest_rays"], st["shadow_rays"]


def _all_budgets_and_streams_agree(monkeypatch, desc, spp):
    want = _frame(monkeypatch, desc, spp, smem=ALL_SHARED, two="0")
    assert want[0][:, :, :3].mean() > 0 and want[2] > 0
    bad = []
    for smem in (ALL_SHARED, "12", "3", "1"):
        for two in ("0", "1"):
            img, closest, shadow = _frame(monkeypatch, desc, spp, smem=smem, two=two)
            if not (np.array_equal(img, want[0]) and closest == want[1] and shadow == want[2]):
                bad.append(f"MFX_STACK_SMEM={smem} MFX_TWO_STREAMS={two}: {int((img != want[0]).any(axis=2).sum())} pixels, "
                           f"rays {closest}/{shadow} against {want[1]}/{want[2]}")
    assert not bad, "frames differ from the all-in-shared one-stream frame: " + "; ".join(bad)


@pytest.mark.gpu
@pytest.mark.parametrize("name,kw", [("haystack", dict(width=160, height=90)), ("c3_renault", dict(width=160, height=90)),
                                     ("spheres", dict(width=160, height=90))])
def test_frames_do_not_depend_on_the_stack_budget_or_the_streams(monkeypatch, name, kw):
    """Fast frames at 16 spp with 1, 3, 12 and all stack entries in shared memory, each on one stream and on two (shadow
    queries of bounce b beside the closest hits of bounce b+1): the same frame and the same ray counts every time."""
    _all_budgets_and_streams_agree(monkeypatch, _desc(name, **kw), 16)


@pytest.mark.gpu
def test_sky_tail_kernel_does_not_depend_on_the_stack_budget(monkeypatch):
    """The sphere sample hands its late bounces to k_f_trace6<TAIL>, which traces and shades a path to its end with one
    stack: one shared entry must render the default frame."""
    desc = scenes.random_scene(width=160, height=80)
    want = _frame(monkeypatch, desc, 8)
    got = _frame(monkeypatch, desc, 8, smem="1")
    assert np.array_equal(got[0], want[0]) and got[1:] == want[1:]


@pytest.mark.gpu
@pytest.mark.parametrize("smem", ["12", "1"])
def test_progressive_film_on_two_streams_equals_one_stream(monkeypatch, smem):
    """Film.GetFrame(integrator, 1) frame after frame (the reference's own render loop: frames of one sample, short
    enough for the two-stream mode) must give the targets a one-stream run gives."""
    from mafrixraytracing_b200 import Scene, CudaPixelIntegrator, Film, FAST_F32
    desc = _haystack(width=160, height=90)
    monkeypatch.setenv("MFX_STACK_SMEM", smem)
    targets = {}
    for two in ("0", "1"):
        monkeypatch.setenv("MFX_TWO_STREAMS", two)
        s = Scene(desc)
        film = Film(s)
        integ = CudaPixelIntegrator(s, precision=FAST_F32, seed=5)
        targets[two] = [film.GetFrame(integ, 1).copy() for _ in range(4)]
        s.close()
    for k, (a, b) in enumerate(zip(targets["1"], targets["0"])):
        assert np.array_equal(a, b), f"frame {k}: {int((a != b).any(axis=2).sum())} pixels differ"


@pytest.mark.gpu
def test_exact_frames_with_one_shared_stack_entry(monkeypatch, goldens):
    """The exact precision sends its closest-hit queries through k_h_trace on the own tree: with one shared entry
    (everything else in the spill columns) its frames must still be the oracle's, bit for bit."""
    from mafrixraytracing_b200 import Scene, CudaPixelIntegrator, EXACT_F64
    from oracle import oracle
    from tests.golden.make_goldens import IMAGES, builder
    monkeypatch.setenv("MFX_STACK_SMEM", "1")
    desc = _haystack(width=48, height=27)
    got = CudaPixelIntegrator(Scene(desc), precision=EXACT_F64, seed=2).Sample(2)
    assert np.array_equal(got[:, :, :3], oracle.OracleScene(desc).sample(2, seed=2)[:, :, :3])
    kw, spp, seed = IMAGES["c3_renault"]
    tex = CudaPixelIntegrator(Scene(builder("c3_renault")(**kw)), precision=EXACT_F64, seed=seed).Sample(spp)
    assert np.array_equal(tex[:, :, :3], goldens["image/c3_renault/rgb"])


@pytest.mark.gpu
@pytest.mark.parametrize("smem", ["64", "1000"])
def test_any_stack_budget_renders(monkeypatch, smem):
    """C3's tree wants 51 entries, more than 48 KB of shared memory holds at 128 threads: a larger budget is capped
    there (the rest spills) instead of failing at launch, and renders the default frame."""
    desc = scenes.c3_renault(width=160, height=90)
    want = _frame(monkeypatch, desc, 4)
    got = _frame(monkeypatch, desc, 4, smem=smem)
    assert np.array_equal(got[0], want[0]) and got[1:] == want[1:]


@pytest.mark.gpu
def test_debug_build_checks_every_spill_index():
    """libmafrix_cuda_dbg.so bounds-checks every stack index the kernels compute (Sample and the seams fail on a
    violation): with one shared entry, fast and exact frames and the closest-hit (id-exact and f32) and any-hit seams of
    the haystack must pass."""
    dbg = os.path.join(ROOT, "mafrixraytracing_b200", "libmafrix_cuda_dbg.so")
    if not os.path.exists(dbg):
        subprocess.check_call(["make", "-C", os.path.join(ROOT, "mafrixraytracing_b200", "csrc"), "-s", "DEBUG=1"])
    code = ("import os\n"
            "import numpy as np\n"
            "from mafrixraytracing_b200 import _lib, Scene, CudaPixelIntegrator, EXACT_F64, FAST_F32\n"
            "from tests.test_gpu_traversal_stack import _haystack\n"
            "assert b'DEBUG CHECKS' in _lib.load().mfx_version()\n"
            "s = Scene(_haystack(width=64, height=36))\n"
            "for prec in (FAST_F32, EXACT_F64):\n"
            "    assert np.isfinite(CudaPixelIntegrator(s, precision=prec, seed=1).Sample(2)).all()\n"
            "rng = np.random.default_rng(0)\n"
            "org = rng.uniform(-2, 2, (20000, 3))\n"
            "d = rng.normal(size=(20000, 3)); d /= np.linalg.norm(d, axis=1)[:, None]\n"
            "s.Hit(org, d, 1e-6, 1e8, precision=FAST_F32)\n"
            "s.Hit(org, d, 1e-6, 2.0, precision=FAST_F32, any_hit=True)\n"
            "os.environ['MFX_F32_PRIMARY'] = '1'\n"
            "s.Hit(org, d, 1e-6, 1e8, precision=FAST_F32)\n"
            "print('spill ok')\n")
    env = dict(os.environ, MFX_LIB=dbg, MFX_STACK_SMEM="1")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "spill ok" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]
