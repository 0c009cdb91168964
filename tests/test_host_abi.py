"""CPU-side checks of the product: the C-ABI library loads and exports every symbol the header
declares, ctypes layouts equal the C ones, the host reproductions (PinholeCamera, Bvh.Build,
tile ownership) agree with the oracle, and compute entry points FAIL LOUDLY without a GPU."""
import ctypes as C
import os
import re
import subprocess
import tempfile

import numpy as np
import pytest

from mafrixraytracing_b200 import _lib, scenes, Bvh, PinholeCamera, Scene, MafrixError
from mafrixraytracing_b200.scene import NODE_DTYPE, make_prims, sphere_prims
from mafrixraytracing_b200 import dist as mdist
from oracle import oracle
from tests.conftest import ROOT, have_gpu

HEADER = os.path.join(ROOT, "include", "mafrix_cuda.h")


def test_library_exports_every_declared_symbol():
    text = open(HEADER).read()
    declared = set(re.findall(r"MFX_API\s+[\w\s\*]+?\b(mfx_\w+)\s*\(", text))
    assert len(declared) >= 24
    assert declared == set(_lib.SYMBOLS), declared ^ set(_lib.SYMBOLS)
    raw = C.CDLL(_lib.LIB_PATH)
    for name in declared:
        assert getattr(raw, name) is not None
    assert b"mafrix_cuda" in _lib.load().mfx_version()


def test_ctypes_layouts_match_the_header():
    src = r'''
#include <stdio.h>
#include <stddef.h>
#include "mafrix_cuda.h"
int main(void) {
  printf("%zu %zu %zu %zu %zu %zu %zu %zu %zu %zu %zu %zu %zu %zu\n", sizeof(MfxPrim), sizeof(MfxMaterial), sizeof(MfxBvhNode),
         sizeof(MfxAreaLight), sizeof(MfxCamera), sizeof(MfxSceneDesc), sizeof(MfxSampleParams), sizeof(MfxStats),
         offsetof(MfxSceneDesc, light), offsetof(MfxStats, ms_total), sizeof(MfxLensCamera), sizeof(MfxSkyTracer),
         offsetof(MfxSkyTracer, perlin_perm), offsetof(MfxSceneDesc, sky));
  return 0; }
'''
    with tempfile.TemporaryDirectory() as td:
        open(os.path.join(td, "s.c"), "w").write(src)
        subprocess.check_call(["/usr/bin/gcc", "-I", os.path.join(ROOT, "include"), "-o", os.path.join(td, "s"), os.path.join(td, "s.c")])
        got = [int(x) for x in subprocess.check_output([os.path.join(td, "s")]).split()]
    from mafrixraytracing_b200.scene import PRIM_DTYPE, MATERIAL_DTYPE
    want = [PRIM_DTYPE.itemsize, MATERIAL_DTYPE.itemsize, NODE_DTYPE.itemsize, C.sizeof(_lib.MfxAreaLight),
            C.sizeof(_lib.MfxCamera), C.sizeof(_lib.MfxSceneDesc), C.sizeof(_lib.MfxSampleParams), C.sizeof(_lib.MfxStats),
            _lib.MfxSceneDesc.light.offset, _lib.MfxStats.ms_total.offset, C.sizeof(_lib.MfxLensCamera),
            C.sizeof(_lib.MfxSkyTracer), _lib.MfxSkyTracer.perlin_perm.offset, _lib.MfxSceneDesc.sky.offset]
    assert got == want


def _build_check_own_tree(tmp_path):
    exe = str(tmp_path / "check_own_tree")
    csrc = os.path.join(ROOT, "mafrixraytracing_b200", "csrc")
    subprocess.check_call(["/usr/bin/g++", "-std=c++17", "-O2", "-pthread", "-I", "/usr/local/cuda/include", "-I", csrc, "-o", exe,
                           os.path.join(ROOT, "tests", "native", "check_own_tree.cpp"), os.path.join(csrc, "mfx_build.cpp")])
    return exe


def test_own_tree_builder_is_a_valid_bvh(tmp_path):
    """The fast path's own SAH tree (csrc/mfx_build.cpp) compiled for the host alone and checked structurally: every
    slot exactly once, every stored box contains its subtree, leaves <= 4, links and depth consistent -- for random
    boxes, coincident boxes (no centroid spread to split on) and a few huge boxes among many small ones."""
    exe = _build_check_own_tree(tmp_path)
    for n, mode in [(1, 0), (2, 0), (3, 0), (5, 0), (17, 0), (1000, 0), (150000, 0), (3000, 1), (5000, 2)]:
        out = subprocess.check_output([exe, str(n), str(mode)], text=True)
        assert out.startswith(f"ok n={n} mode={mode}"), out
    # the reinsertion pass (sah_reinsert: default 2 passes over the 32768 largest subtrees) moves whole subtrees: valid
    # trees for any number of passes and any bound on the subtrees moved, and a SAH cost that does not rise
    def cost(n, mode, **env):
        out = subprocess.check_output([exe, str(n), str(mode)], text=True, env=dict(os.environ, **env))
        assert out.startswith(f"ok n={n} mode={mode}"), (env, out)
        return float(out.split("cost=")[1].split()[0])
    for n, mode in [(5, 0), (17, 0), (1000, 0), (40000, 0), (3000, 1), (5000, 2)]:
        base = cost(n, mode, MFX_TREE_OPT="0")
        for env in (dict(MFX_TREE_OPT="1"), dict(MFX_TREE_OPT="4"), dict(MFX_TREE_OPT="2", MFX_TREE_OPT_NODES="50"), dict(MFX_TREE_OPT="2", MFX_TREE_OPT_MAX="10")):
            assert cost(n, mode, **env) <= base * 1.02, (n, mode, env)
    assert cost(5000, 2, MFX_TREE_OPT="2") < 0.97 * cost(5000, 2, MFX_TREE_OPT="0")         # a few huge boxes among small ones: the pass pays
    # coincident boxes: every position costs the same -- nothing may move (a non-strict rule chains the tree: depth 341)
    out = subprocess.check_output([exe, "3000", "1"], text=True, env=dict(os.environ, MFX_TREE_OPT="3"))
    assert int(out.split("depth=")[1].split()[0]) <= 8, out
    # the greedy collapse of round 1 (MFX_COLLAPSE_DP=0) and another record cost must give valid trees too
    for dp in ("0", "250"):
        for n, mode in [(1, 0), (3, 0), (5, 0), (17, 0), (1000, 0), (40000, 0), (3000, 1), (5000, 2)]:
            out = subprocess.check_output([exe, str(n), str(mode)], text=True, env=dict(os.environ, MFX_COLLAPSE_DP=dp))
            assert out.startswith(f"ok n={n} mode={mode}"), (dp, out)


def test_own_tree_does_not_depend_on_the_fork_depth(tmp_path):
    """The builder forks its top levels over threads.  The tree must be the same for any fork depth and any schedule of
    those threads: the spot mesh of C2 has many subtrees of equal area, where the reinsertion pass breaks ties by node
    index, so node indices handed out in the threads' order would change the tree from run to run."""
    exe = _build_check_own_tree(tmp_path)
    tris = []
    for p in scenes.c2_spot().prims:
        tris.append(p["v"][:9])
        if p["kind"] == 1:                                    # a Rect is two triangles, as the fast path slots it
            tris.append(np.concatenate([p["v"][0:3], p["v"][6:9], p["v"][9:12]]))
    path = str(tmp_path / "tris.bin")
    np.array(tris, np.float64).tofile(path)
    trees = set()
    for depth in ("0", "1", "2", "3", "3", "5", "5", "5"):
        out = subprocess.check_output([exe, str(len(tris)), "3", path], text=True, env=dict(os.environ, MFX_BVH_BUILD_PAR_DEPTH=depth))
        assert out.startswith(f"ok n={len(tris)} mode=3"), out
        trees.add(out.split("tree=")[1].split()[0])
    assert len(trees) == 1, trees


def test_fsharp_shim_offsets_match_the_header():
    """host/fsharp/MafrixCuda.fs writes the C structs into unmanaged memory by hand (no .NET here to compile it):
    every offset it uses must be the header's."""
    fields = [("MfxPrim", "kind"), ("MfxPrim", "material"), ("MfxPrim", "v"), ("MfxMaterial", "albedo"), ("MfxMaterial", "fuzz"),
              ("MfxMaterial", "ei"), ("MfxMaterial", "et"), ("MfxBvhNode", "pmax"), ("MfxBvhNode", "first"), ("MfxBvhNode", "count"),
              ("MfxSceneDesc", "n_prims"), ("MfxSceneDesc", "materials"), ("MfxSceneDesc", "n_materials"), ("MfxSceneDesc", "nodes"),
              ("MfxSceneDesc", "n_node_slots"), ("MfxSceneDesc", "indices"), ("MfxSceneDesc", "light"), ("MfxSceneDesc", "camera"),
              ("MfxSceneDesc", "width"), ("MfxSceneDesc", "height"), ("MfxSceneDesc", "max_depth"), ("MfxSceneDesc", "integrator"),
              ("MfxSceneDesc", "sky"), ("MfxAreaLight", "normal"), ("MfxAreaLight", "color"), ("MfxCamera", "topleft"), ("MfxCamera", "right"), ("MfxCamera", "down"),
              ("MfxSampleParams", "seed"), ("MfxSampleParams", "first_sample"), ("MfxSampleParams", "flags")]
    body = "".join(f'  printf("%zu\\n", offsetof({t}, {f}));\n' for t, f in fields)
    src = '#include <stdio.h>\n#include <stddef.h>\n#include "mafrix_cuda.h"\nint main(void) {\n' + body + \
          '  printf("%zu %zu %zu %zu %zu\\n", sizeof(MfxPrim), sizeof(MfxMaterial), sizeof(MfxBvhNode), sizeof(MfxSceneDesc), sizeof(MfxSampleParams));\n  return 0; }\n'
    with tempfile.TemporaryDirectory() as td:
        open(os.path.join(td, "s.c"), "w").write(src)
        subprocess.check_call(["/usr/bin/gcc", "-I", os.path.join(ROOT, "include"), "-o", os.path.join(td, "s"), os.path.join(td, "s.c")])
        out = subprocess.check_output([os.path.join(td, "s")]).split()
    off = {tf: int(v) for tf, v in zip(fields, out)}
    sizes = [int(v) for v in out[len(fields):]]
    assert sizes == [104, 56, 56, 320, 40]
    want = {("MfxPrim", "kind"): 0, ("MfxPrim", "material"): 4, ("MfxPrim", "v"): 8, ("MfxMaterial", "albedo"): 8, ("MfxMaterial", "fuzz"): 32,
            ("MfxMaterial", "ei"): 40, ("MfxMaterial", "et"): 48, ("MfxBvhNode", "pmax"): 24, ("MfxBvhNode", "first"): 48, ("MfxBvhNode", "count"): 52,
            ("MfxSceneDesc", "n_prims"): 8, ("MfxSceneDesc", "materials"): 16, ("MfxSceneDesc", "n_materials"): 24, ("MfxSceneDesc", "nodes"): 32,
            ("MfxSceneDesc", "n_node_slots"): 40, ("MfxSceneDesc", "indices"): 48, ("MfxSceneDesc", "light"): 56, ("MfxSceneDesc", "camera"): 200,
            ("MfxSceneDesc", "width"): 296, ("MfxSceneDesc", "height"): 300, ("MfxSceneDesc", "max_depth"): 304, ("MfxSceneDesc", "integrator"): 308,
            ("MfxSceneDesc", "sky"): 312, ("MfxAreaLight", "normal"): 96, ("MfxAreaLight", "color"): 120, ("MfxCamera", "topleft"): 24, ("MfxCamera", "right"): 48, ("MfxCamera", "down"): 72,
            ("MfxSampleParams", "seed"): 8, ("MfxSampleParams", "first_sample"): 16, ("MfxSampleParams", "flags"): 32}
    assert off == want
    # ... and the shim really uses those numbers (the table above is what its comments and writes state)
    fs = open(os.path.join(ROOT, "host", "fsharp", "MafrixCuda.fs")).read()
    for needle in ("AllocHGlobal(104 * hs.Length)", "AllocHGlobal 320", "WriteIntPtr(d, 312, 0n)", "WriteInt32(d, 296, width)", "WriteInt32(d, 300, height)",
                   "WriteInt32(d, 304, maxDepth)", "WriteInt32(d, 308,", "Interop.wpt d 200 cam.position", "Interop.wpt d 224 cam.topleft",
                   "Interop.wd d 248 cam.coord.right.x", "Interop.wd d 272 cam.coord.down.x", "Interop.wd d 152 light.normal.x",
                   "Interop.wd d 176 light.color.r", "WriteIntPtr(d, 48, pIdx)", "WriteInt32(mem, b + 48, n.first)", "wd mem (b + 32) fuzz"):
        assert needle in fs, needle
    import re
    for sym in re.findall(r"extern \w+ (mfx_\w+)\(", fs):
        assert sym in _lib.SYMBOLS, sym


@pytest.mark.parametrize("pos,dir,fov,aspect", [((0, 1, 3), (0, 0, -1), 120.0, 1.0), ((4.5, 1.6, 5.5), (-0.62, -0.18, -0.76), 120.0, 16 / 9),
                                                ((13, 2, 3), (-13, -2, -3), 90.0, 4 / 3), ((0, 0.1, -2.6), (0, 0, 1), 37.5, 2.0)])
def test_camera_matches_oracle_bitwise(pos, dir, fov, aspect):
    cam = PinholeCamera(pos, dir, fov, aspect)
    assert np.array_equal(cam.derived(), oracle.camera_pinhole(pos, dir, fov, aspect))
    o, d = cam.GetRay(0.5, 0.5)
    assert abs(np.linalg.norm(d) - 1) < 1e-15


def _same_tree(desc):
    b = Bvh.Build(desc.prims)
    nodes, idx = oracle.OracleScene(desc).bvh()
    assert np.array_equal(idx, b.indices)
    assert np.array_equal(nodes.view(np.uint8), b.nodes.view(np.uint8))
    return b


@pytest.mark.parametrize("name,kw", [("cornell", {}), ("c1_cube", {}), ("c2_spot", dict(width=8, height=8)),
                                     ("c3_renault", dict(width=8, height=8)), ("c4_spheres", dict(width=8, height=8, grid=40))])
def test_bvh_build_matches_oracle(name, kw):
    b = _same_tree(scenes.WORKLOADS[name](**kw))
    assert b.nodes[0]["count"] == len(b.indices)


def test_bvh_build_ties_and_mixed_primitives():
    d = scenes.cornell(width=8, height=8)
    rng = np.random.default_rng(9)
    tris = make_prims(40)
    tris["v"][:, :9] = np.repeat(rng.uniform(-1, 1, (8, 9)), 5, axis=0)          # 5 exact duplicates each -> key ties
    sph = sphere_prims(rng.uniform(-1, 1, (11, 3)), rng.uniform(0.05, 0.3, 11), 0)
    d.prims = np.concatenate([d.prims, tris, sph])
    _same_tree(d)


def test_bvh_build_rejects_bad_arguments():
    lib = _lib.load()
    prims = scenes.cornell(width=8, height=8).prims
    nodes = np.zeros(2 * len(prims) - 1, NODE_DTYPE)
    idx = np.zeros(len(prims), np.int32)
    assert lib.mfx_bvh_build(_lib.ptr(prims), len(prims), _lib.ptr(nodes), len(nodes) - 1, _lib.ptr(idx)) == -1
    assert b"2n-1" in lib.mfx_last_error()
    assert lib.mfx_bvh_build(None, 3, _lib.ptr(nodes), 5, _lib.ptr(idx)) == -1
    bad = prims.copy()
    bad["kind"][0] = 7
    assert lib.mfx_bvh_build(_lib.ptr(bad), len(bad), _lib.ptr(nodes), len(nodes), _lib.ptr(idx)) == -1


def test_scene_create_validates_before_touching_the_device():
    d = scenes.cornell(width=8, height=8)
    d.prims = d.prims.copy()
    d.prims["material"][3] = 99
    with pytest.raises(MafrixError) as e:
        Scene(d)
    assert e.value.code == -1 and "material" in str(e.value)
    d2 = scenes.cornell(width=8, height=8)
    d2.max_depth = 64
    with pytest.raises(MafrixError) as e:
        Scene(d2)
    assert e.value.code == -5
    # the sphere sample (MFX_SKY_TRACER): spheres only, its own material kinds, the noise tables when a material needs them
    d3 = scenes.random_scene(width=8, height=8)
    d3.prims = d3.prims.copy()
    d3.prims["kind"][0] = 0
    with pytest.raises(MafrixError) as e:
        Scene(d3)
    assert e.value.code == -5 and "spheres" in str(e.value)
    d4 = scenes.random_scene(width=8, height=8)
    d4.sky.ranfloat = None
    with pytest.raises(MafrixError) as e:
        Scene(d4)
    assert e.value.code == -1 and "Perlin" in str(e.value)
    d5 = scenes.random_scene(width=8, height=8)
    d5.sky = None
    with pytest.raises(MafrixError) as e:
        Scene(d5)
    assert e.value.code == -1 and "sky" in str(e.value)
    d6 = scenes.cornell(width=8, height=8)
    d6.materials = d6.materials.copy()
    d6.materials["kind"][0] = 3                     # Dielectric only exists under the sky tracer
    with pytest.raises(MafrixError) as e:
        Scene(d6)
    assert e.value.code == -1
    # a caller-supplied Bvh is indexed by the flatteners and the kernels: malformed ones are refused, not dereferenced
    d7 = scenes.cornell(width=8, height=8)
    good = Bvh.Build(d7.prims)
    for what, breakit in (("permutation", lambda b: b.indices.__setitem__(2, b.indices[3])),
                          ("permutation", lambda b: b.indices.__setitem__(0, len(d7.prims) + 5)),
                          ("covers", lambda b: b.nodes["first"].__setitem__(1, -3)),
                          ("cover", lambda b: b.nodes["count"].__setitem__(2, 1))):
        bad = Bvh(good.nodes.copy(), good.indices.copy())
        breakit(bad)
        with pytest.raises(MafrixError) as e:
            Scene(d7, bvh=bad)
        assert e.value.code == -1 and what in str(e.value), str(e.value)
    with pytest.raises(MafrixError) as e:
        Scene(d7, bvh=Bvh(good.nodes[:-2].copy(), good.indices.copy()))
    assert e.value.code == -1 and "2n-1" in str(e.value)


@pytest.mark.skipif(have_gpu(), reason="a CUDA device is present")
def test_no_cpu_fallback_without_a_gpu():
    lib = _lib.load()
    assert lib.mfx_device_count() == 0
    assert lib.mfx_init(0) == -2 and b"no CPU fallback" in lib.mfx_last_error()
    with pytest.raises(MafrixError) as e:
        Scene(scenes.cornell(width=8, height=8))
    assert e.value.code == -2


@pytest.mark.parametrize("w,h,tile,world", [(1920, 1080, 64, 8), (300, 300, 64, 2), (17, 5, 4, 3), (64, 64, 64, 4), (100, 37, 16, 1)])
def test_tile_map_partitions_the_frame(w, h, tile, world):
    seen = np.zeros(w * h, np.int32)
    sizes = []
    for r in range(world):
        pix = mdist.tile_pixels(w, h, tile, r, world)
        seen[pix] += 1
        sizes.append(len(pix))
        ty, tx = (pix // w) // tile, (pix % w) // tile
        assert ((ty * ((w + tile - 1) // tile) + tx) % world == r).all()
    assert (seen == 1).all()
    if w * h >= world * tile * tile * 8:
        assert max(sizes) - min(sizes) <= 2 * tile * tile
    lib = _lib.load()
    n = C.c_int32()
    assert lib.mfx_tile_map(w, h, tile, world, world, None, C.byref(n)) == -1


@pytest.mark.parametrize("w,h,stripe,world", [(1920, 1080, 16, 8), (300, 300, 16, 3), (70, 33, 8, 2), (50, 7, 16, 5), (16, 4, 16, 4)])
def test_stripe_map_partitions_the_frame(w, h, stripe, world):
    """Column-stripe ownership (MFX_SAMPLE_STRIPES, what mfx_multi_sample and the torchrun path shard by): every pixel
    has one owner, stripe c belongs to rank c % world, and the local order is stripe after stripe, row-major inside."""
    seen = np.zeros(w * h, int)
    for r in range(world):
        pix = mdist.stripe_pixels(w, h, stripe, r, world)
        seen[pix] += 1
        x, y = pix % w, pix // w
        assert ((x // stripe) % world == r).all()
        # the arithmetic the kernels use (pixel_of in mfx_device.cuh), restated
        pl = np.arange(len(pix))
        per = stripe * h
        ls, rem = pl // per, pl % per
        x0 = (ls * world + r) * stripe
        wl = np.minimum(stripe, w - x0)
        assert np.array_equal(y, rem // wl) and np.array_equal(x, x0 + rem % wl)
    assert (seen == 1).all()
    n = C.c_int32()
    assert _lib.load().mfx_stripe_map(w, h, stripe, world, world, None, C.byref(n)) == -1


def test_workload_builders_match_the_configs():
    d = scenes.c2_spot()
    assert (d.width, d.height, d.max_depth, d.integrator, len(d.prims)) == (1920, 1080, 5, 0, 5858)
    d = scenes.c3_renault()
    assert (d.width, d.height, d.integrator, len(d.prims)) == (1920, 1080, 1, 36997)
    assert set(np.unique(d.prims["material"])) == {0, 1, 2}
    d = scenes.c1_cube()
    assert (d.width, d.height, d.max_depth, len(d.prims)) == (640, 480, 5, 17)
    d = scenes.cornell()
    assert (d.width, d.height, d.max_depth) == (300, 300, 3) and (d.prims["kind"] == 1).all()
    # every room/box surface faces the way the unflipped-normal integrator needs (quirk Q4)
    v = d.prims["v"].reshape(-1, 4, 3)
    n = np.cross(v[:, 1] - v[:, 0], v[:, 2] - v[:, 0])
    assert n[0][1] > 0 and n[1][1] < 0 and n[2][2] > 0 and n[3][0] < 0 and n[4][0] > 0


def test_cpp_host_driver_builds_and_fails_loudly_without_gpu():
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "host"), "-s"])
    exe = os.path.join(ROOT, "host", "render_test")
    assert os.path.exists(exe)
    if not have_gpu():
        r = subprocess.run([exe, "--frames", "1"], capture_output=True, text=True)
        assert r.returncode == 1 and "no CPU fallback" in r.stderr
