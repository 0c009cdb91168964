"""Parity of the CUDA path (through the C ABI) against the CPU oracle and the committed goldens.

Bars (BASELINE.json north_star):
  * MFX_EXACT_F64: primitive ids, t AND radiance bit-exact (integer/index work: bit-exact;
    the f64 path reproduces the reference's rounding sequence, so we hold it to bit-exact too);
  * MFX_FAST_F32 : primary-hit buffers (ids AND t) bit-exact too -- bounce 0 and the closest-hit seams run the
    id-exact hybrid traversal (mfx_hybrid.cu: f32 boxes, f64 primitive tests, the reference's tie rules); with
    MFX_SAMPLE_F32_PRIMARY / MFX_F32_PRIMARY=1 (f32 primitive tests everywhere, the round-1 kernel) ids agree except
    on <= 2e-4 of the rays and t within 1e-4 relative; images within a stated relative RMSE of the exact frame at
    matched spp and seeds.
"""
import hashlib
import os

import numpy as np
import pytest

from mafrixraytracing_b200 import (scenes, Scene, CudaPixelIntegrator, Film, Bvh, MafrixError, EXACT_F64, FAST_F32,
                                   PATH_INTEGRATOR, NEW_PATH_TRACER)
from mafrixraytracing_b200 import _lib
from mafrixraytracing_b200.scene import (AreaLight, PinholeCamera, SceneDesc, make_materials, make_prims, sphere_prims,
                                         rect_prim)
from oracle import oracle

pytestmark = pytest.mark.gpu
BIG = 99999999.


def _sha(a):
    return np.frombuffer(hashlib.sha256(np.ascontiguousarray(a).tobytes()).digest(), dtype=np.uint8)


def _desc(name, **kw):
    base = name.replace("_small", "")
    return (scenes.c4_spheres if base == "spheres" else scenes.WORKLOADS[base])(**kw)


# ------------------------------------------------------------------ primary-hit buffers
@pytest.mark.parametrize("name,kw", [("cornell", {}), ("c1_cube", {}), ("c2_spot_small", dict(width=480, height=270)),
                                     ("c3_renault_small", dict(width=480, height=270))])
def test_exact_primary_bit_exact_vs_oracle_and_goldens(goldens, name, kw):
    desc = _desc(name, **kw)
    s = Scene(desc)
    prim, t = s.TracePrimary(precision=EXACT_F64)
    oprim, ot = oracle.OracleScene(desc).trace_primary()
    assert np.array_equal(prim, oprim) and np.array_equal(t, ot)
    assert np.array_equal(prim, goldens[f"primary/{name}/prim"])
    assert np.array_equal(_sha(t), goldens[f"primary/{name}/sha_t"])


@pytest.mark.parametrize("name", ["c2_spot", "c3_renault"])
def test_exact_primary_full_size_matches_golden_checksums(goldens, name):
    s = Scene(_desc(name))                      # 1920x1080, BASELINE configs[1] / [2]
    prim, t = s.TracePrimary(precision=EXACT_F64)
    assert int((prim >= 0).sum()) == int(goldens[f"primary/{name}/hits"])
    assert np.array_equal(_sha(prim), goldens[f"primary/{name}/sha_prim"])
    assert np.array_equal(_sha(t), goldens[f"primary/{name}/sha_t"])


@pytest.mark.parametrize("name,kw", [("cornell", {}), ("c1_cube", {}), ("c2_spot", dict(width=640, height=360)),
                                     ("c3_renault", dict(width=640, height=360)), ("spheres", dict(width=640, height=360, grid=40))])
def test_fast_primary_is_bit_exact(name, kw):
    """north_star: primary-hit ids bit-exact.  The throughput path's bounce-0 kernel (hybrid: own SAH tree, f32 boxes,
    f64 leaf tests) must return the oracle's primitive AND its f64 t on every one of 300 k jittered rays."""
    desc = _desc(name, **kw)
    s = Scene(desc)
    rng = np.random.default_rng(4)
    uv = rng.random((300000, 2))                # jittered rays: pixel centres sit on quad diagonals
    oprim, ot = oracle.OracleScene(desc).trace_primary(uv)
    prim, t = s.TracePrimary(uv, precision=FAST_F32)
    assert int((prim != oprim).sum()) == 0, f"{int((prim != oprim).sum())} primary ids differ from the oracle"
    assert np.array_equal(t, ot)
    eprim, et = s.TracePrimary(uv, precision=EXACT_F64)
    assert np.array_equal(eprim, oprim) and np.array_equal(et, ot)


@pytest.mark.parametrize("name", ["c2_spot", "c3_renault"])
def test_fast_primary_full_size_matches_golden_checksums(goldens, name):
    """The 1920x1080 pixel-centre buffers of BASELINE configs[1] / [2] through the throughput path's primary kernel
    hash to the oracle's committed checksums (pixel centres sit exactly on quad diagonals and shared edges: ties)."""
    s = Scene(_desc(name))
    prim, t = s.TracePrimary(precision=FAST_F32)
    assert int((prim >= 0).sum()) == int(goldens[f"primary/{name}/hits"])
    assert np.array_equal(_sha(prim), goldens[f"primary/{name}/sha_prim"])
    assert np.array_equal(_sha(t), goldens[f"primary/{name}/sha_t"])


@pytest.mark.parametrize("name,kw", [("cornell", {}), ("c2_spot", dict(width=640, height=360)), ("c3_renault", dict(width=640, height=360))])
def test_f32_primary_ids_and_t_tolerance(monkeypatch, name, kw):
    """The f32 primitive tests (what bounces >= 1 use; bounce 0 only on request): ids within 2e-4, t within 1e-4."""
    monkeypatch.setenv("MFX_F32_PRIMARY", "1")
    desc = _desc(name, **kw)
    s = Scene(desc)
    rng = np.random.default_rng(4)
    uv = rng.random((300000, 2))
    oprim, ot = oracle.OracleScene(desc).trace_primary(uv)
    prim, t = s.TracePrimary(uv, precision=FAST_F32)
    mism = (prim != oprim).mean()
    assert mism <= 2e-4, f"fast primary id mismatch rate {mism:.2e}"
    both = (prim == oprim) & (oprim >= 0)
    assert (np.abs(t[both] - ot[both]) <= 1e-4 * np.abs(ot[both])).all()      # north_star: t within 1e-4 relative


def test_hybrid_hands_the_unprovable_rays_to_the_exact_walk():
    """Rays the hybrid kernel cannot clear by its one-box argument -- a zero direction component, a winner beyond
    tMax (quirk Q2), the tie and Rect quirks -- must come back from k_h_fixup with the oracle's answer."""
    desc = _desc("cornell", width=64, height=64)
    s, o = Scene(desc), oracle.OracleScene(desc)
    rng = np.random.default_rng(11)
    n = 20000
    org = rng.uniform(-0.9, 0.9, (n, 3)); org[:, 1] += 1.0
    d = rng.normal(size=(n, 3))
    d[: n // 2, rng.integers(0, 3)] = 0.0                       # axis-parallel: the 0/0 family of AABB.hit (quirk Q6)
    d /= np.linalg.norm(d, axis=1)[:, None]
    for tmax in (BIG, 0.7):                                     # tMax-blind triangles: hits beyond tMax survive in all-hit leaves
        op, osub, ot = o.hit(org, d, 1e-6, tmax)
        fp, fsub, ft = s.Hit(org, d, 1e-6, tmax, precision=FAST_F32)
        assert np.array_equal(fp, op) and np.array_equal(fsub, osub) and np.array_equal(ft, ot)
    st = _lib.MfxStats()
    _lib.check(_lib.load().mfx_get_stats(s._h, __import__("ctypes").byref(st)))
    assert st.hybrid_fixups >= n // 2                           # the axis-parallel half went through the exact walk


# ------------------------------------------------------------------ Bvh.Hit seam
@pytest.mark.parametrize("name,kw", [("cornell", {}), ("c1_cube", {}), ("c2_spot", dict(width=8, height=8)),
                                     ("c3_renault", dict(width=8, height=8)), ("spheres", dict(width=8, height=8, grid=30))])
def test_bvh_hit_closest_and_shadow(monkeypatch, name, kw):
    desc = _desc(name, **kw)
    s, o = Scene(desc), oracle.OracleScene(desc)
    rng = np.random.default_rng(3)
    n = 100000
    org = rng.uniform(-3, 3, (n, 3))
    if name == "spheres":
        org[:, 1] = rng.uniform(0.05, 3, n)
    d = rng.normal(size=(n, 3))
    d /= np.linalg.norm(d, axis=1)[:, None]
    op, osub, ot = o.hit(org, d, 1e-6, BIG)
    gp, gsub, gt = s.Hit(org, d, 1e-6, BIG, precision=EXACT_F64)
    assert np.array_equal(gp, op) and np.array_equal(gsub, osub) and np.array_equal(gt, ot)
    fp, fsub, ft = s.Hit(org, d, 1e-6, BIG, precision=FAST_F32)          # closest hit: the id-exact hybrid kernel
    assert np.array_equal(fp, op) and np.array_equal(fsub, osub) and np.array_equal(ft, ot)
    monkeypatch.setenv("MFX_F32_PRIMARY", "1")                           # the f32 primitive tests of bounces >= 1
    fp, fsub, ft = s.Hit(org, d, 1e-6, BIG, precision=FAST_F32)
    monkeypatch.delenv("MFX_F32_PRIMARY")
    assert (fp != op).mean() <= 3e-4
    same = (fp == op) & (op >= 0)
    # random origins can sit arbitrarily close to a surface: f32 absolute error ~ a few ulp of the
    # scene extent (6 units -> ~5e-7 each op), so the relative bar gets an absolute floor here
    # (the sphere scene holds the r=1000 ground sphere: ulp(1000) = 6e-5 bounds what f32 can resolve)
    # the kernel solves that one in f64, small spheres in f32)
    floor = 5e-5 if name == "spheres" else 2e-5
    bad = np.abs(ft[same] - ot[same]) > 1e-4 * np.abs(ot[same]) + floor
    # an origin within ~1e-6 of a sphere can take the near root in one precision and the far root in
    # the other (same primitive id, t differs by a chord): allowed for at most 1e-4 of the rays
    assert bad.mean() <= (1e-4 if name == "spheres" else 0.0), (bad.sum(), np.abs(ft[same] - ot[same]).max())
    for tmax in (0.5, 2.0):                      # shadow queries (Integrators.fs:44)
        op, _, _ = o.hit(org, d, 1e-6, tmax)
        gp, _, _ = s.Hit(org, d, 1e-6, tmax, precision=EXACT_F64, any_hit=True)
        assert np.array_equal(gp >= 0, op >= 0)
        fp, _, _ = s.Hit(org, d, 1e-6, tmax, precision=FAST_F32, any_hit=True)
        assert ((fp >= 0) != (op >= 0)).mean() <= 3e-4


def test_exact_reproduces_the_quirks():
    # Q1 tie rules, Q2 tMax-blind triangles, Q3 Rect returns tri1 first, Q6 NaN / -0.0 box tests
    def tri(v0, v1, v2):
        p = make_prims(1)
        p["v"][0, :9] = np.concatenate([v0, v1, v2])
        return p

    def scene_of(prims):
        mats = make_materials([("lambert", (0.5, 0.5, 0.5))])
        light = AreaLight(np.array([(-1, 5, 1), (-1, 5, -1), (1, 5, -1), (1, 5, 1)], float), (0, -1, 0), (10, 10, 10))
        desc = SceneDesc(np.concatenate(prims), mats, light, PinholeCamera((0, 0, 5), (0, 0, -1), 120.0, 1.0), 8, 8, 0)
        return Scene(desc), oracle.OracleScene(desc)

    unit = tri((0, 0, 0), (1, 0, 0), (0, 1, 0))
    cases = [
        ([unit] * 8, (0.25, 0.25, 1), (0, 0, -1), 1e-6, BIG),
        ([unit] * 3, (0.25, 0.25, 1), (0, 0, -1), 1e-6, BIG),
        ([tri((0, 0, 0), (1, 0, 1), (0, 1, 0))], (0.1, 0.1, 2), (0, 0, -1), 1e-6, 1.5),
        ([tri((0, 0, 0), (1, 0, 1), (0, 1, 0)), tri((5, 5, 0), (6, 5, 0), (5, 6, 0))], (0.1, 0.1, 2), (0, 0, -1), 1e-6, 1.5),
        ([rect_prim((0, 0, 0), (1, 0, 0), (1, 1, 0), (1, 0.2, 0.5))], (0.8, 0.4, 2), (0, 0, -1), 1e-6, BIG),
        ([unit], (0.0, 0.3, 1), (0, 0, -1), 1e-6, BIG),
        ([unit], (0.25, 0.25, 2), (-0.0, 0.0, -1.0), 1e-6, BIG),
        ([unit], (0.5, 0.3, 1), (-0.5, 0, -1), 1e-6, BIG),
        ([sphere_prims([(0, 0, 0)], 1.0, 0)], (0, 0, 0), (0, 0, -1), 1e-6, BIG),
        ([sphere_prims([(0, 0, 0)], 1.0, 0)], (1, 0, 3), (0, 0, -1), 1e-6, BIG),
    ]
    for prims, org, d, tmin, tmax in cases:
        s, o = scene_of(prims)
        for any_hit in (False, True):
            want = o.hit([org], [d], tmin, tmax)
            got = s.Hit([org], [d], tmin, tmax, precision=EXACT_F64, any_hit=any_hit)
            if any_hit:
                assert (got[0] >= 0) == (want[0] >= 0)
            else:
                assert all(np.array_equal(a, b) for a, b in zip(got, want)), (org, d, got, want)


# ------------------------------------------------------------------ IPixelIntegrator.Sample
@pytest.mark.parametrize("name", ["cornell", "c1_cube", "c2_spot", "c3_renault", "spheres"])
def test_exact_sample_bit_exact_vs_goldens_and_oracle(goldens, name):
    from tests.golden.make_goldens import IMAGES, builder
    kw, spp, seed = IMAGES[name]
    desc = builder(name)(**kw)
    s = Scene(desc)
    integ = CudaPixelIntegrator(s, precision=EXACT_F64, seed=seed)
    tex = integ.Sample(spp)
    assert tex.shape == (desc.width, desc.height, 4) and (tex[:, :, 3] == 1.0).all()
    assert np.array_equal(tex[:, :, :3], goldens[f"image/{name}/rgb"])
    o = oracle.OracleScene(desc)
    ref, st = o.sample(spp, seed=seed, stats=True)
    assert np.array_equal(tex[:, :, :3], ref[:, :, :3])
    assert integ.stats["closest_rays"] == st["closest_rays"] and integ.stats["shadow_rays"] == st["shadow_rays"]
    assert integ.stats["paths"] == desc.width * desc.height * spp


@pytest.mark.parametrize("name,kw,spp,tol", [("cornell", dict(width=150, height=150), 16, 5e-3),
                                             ("c1_cube", dict(width=160, height=120), 16, 5e-3),
                                             ("c2_spot", dict(width=240, height=135), 16, 2e-2)])
def test_fast_sample_tracks_exact_at_matched_seeds(name, kw, spp, tol):
    """Same Philox stream in both precisions (MFX_SAMPLE_REFERENCE_STREAM: the fast path runs the reference's
    rejection loop on the f32 view of the exact stream): most paths take identical decisions, so the f32 frame
    stays within `tol` relative RMSE of the exact frame (stated tolerance, mode A)."""
    desc = _desc(name, **kw)
    s = Scene(desc)
    exact = CudaPixelIntegrator(s, precision=EXACT_F64, seed=5).Sample(spp).copy()
    fast = CudaPixelIntegrator(s, precision=FAST_F32, seed=5).Sample(spp, flags=_lib.SAMPLE_REFERENCE_STREAM).copy()
    rel = np.sqrt(((fast - exact)[:, :, :3] ** 2).mean()) / np.abs(exact[:, :, :3]).mean()
    assert rel <= tol, f"{name}: relative RMSE {rel:.3e}"
    assert abs(fast[:, :, :3].mean() / exact[:, :, :3].mean() - 1) < 2e-3


@pytest.mark.parametrize("name,kw,mode", [("cornell", dict(width=96, height=96), None), ("c2_spot", dict(width=128, height=72), None),
                                          ("c3_renault", dict(width=128, height=72), None),
                                          ("spheres", dict(width=128, height=72, grid=16), None)])
def test_direct_sampler_converges_to_the_rejection_sampler(name, kw, mode):
    """The default fast sampler draws the hemisphere direction / half-ball point / light point directly (one RNG call
    per vertex) instead of the reference's rejection loop (Material.fs:9-14).  Same distributions => same expected
    frame: the difference between the two samplers must be no larger than the difference between two seeds of the
    rejection sampler, and the mean radiance must agree."""
    desc = _desc(name, **kw)
    s = Scene(desc)
    spp = 512
    ra = CudaPixelIntegrator(s, precision=FAST_F32, seed=11).Sample(spp, flags=_lib.SAMPLE_REFERENCE_STREAM).copy()[:, :, :3]
    rb = CudaPixelIntegrator(s, precision=FAST_F32, seed=12).Sample(spp, flags=_lib.SAMPLE_REFERENCE_STREAM).copy()[:, :, :3]
    da = CudaPixelIntegrator(s, precision=FAST_F32, seed=11).Sample(spp).copy()[:, :, :3]
    assert not np.array_equal(da, ra)
    clip = np.percentile(np.abs(ra), 99.5)
    c = lambda x: np.clip(x, -clip, clip)
    noise = np.sqrt(((c(ra) - c(rb)) ** 2).mean())
    err = np.sqrt(((c(da) - c(ra)) ** 2).mean())
    assert err <= 1.1 * noise, f"{name}: direct-vs-rejection {err:.3e} exceeds the seed-to-seed noise {noise:.3e}"
    assert abs(c(da).mean() / c(ra).mean() - 1) < 5e-3, f"{name}: mean radiance {c(da).mean():.5e} vs {c(ra).mean():.5e}"


@pytest.mark.parametrize("name,kw,tol64,tol256", [("c3_renault", dict(width=160, height=90), 0.40, 0.20),
                                                  ("spheres", dict(width=160, height=90, grid=24), 0.19, 0.095)])
def test_fast_sample_mode_b_stated_tolerance(name, kw, tol64, tol256):
    """NewPathTracer scenes have specular chains and 1/|cos| weights: single paths diverge between f32 and f64, so the
    bar is on converged images at matched spp (north_star).  STATED TOLERANCE, 99th-percentile-clipped radiance:
      relative RMSE of the fast frame against the exact frame  <= tol64 at 64 spp, <= tol256 at 256 spp
        (measured 0.34 / 0.17 on Renault, 0.15 / 0.075 on the spheres: it halves per 4x spp -- both renderers converge to
         the same image -- and stays BELOW the exact renderer's own seed-to-seed RMSE, 0.40 / 0.20 and 0.19 / 0.093);
      relative luminance (Rec. 709) of the whole frame within 5e-3 at 64 spp and 2e-3 at 256 spp (measured <= 3.2e-3 / 8e-4)."""
    desc = _desc(name, **kw)
    s = Scene(desc)
    rel = {}
    for spp, tol, ltol in ((64, tol64, 5e-3), (256, tol256, 2e-3)):
        ea = CudaPixelIntegrator(s, precision=EXACT_F64, seed=5).Sample(spp).copy()[:, :, :3]
        eb = CudaPixelIntegrator(s, precision=EXACT_F64, seed=6).Sample(spp).copy()[:, :, :3]
        fa = CudaPixelIntegrator(s, precision=FAST_F32, seed=5).Sample(spp).copy()[:, :, :3]
        # robust statistics: heavy-tailed fireflies make plain RMSE meaningless here
        clip = np.percentile(ea, 99.0)
        c = lambda x: np.clip(x, -clip, clip)
        lum = lambda x: (c(x) * [0.2126, 0.7152, 0.0722]).sum(-1).mean()
        mean = np.abs(c(ea)).mean()
        noise = np.sqrt(((c(ea) - c(eb)) ** 2).mean()) / mean
        rel[spp] = np.sqrt(((c(fa) - c(ea)) ** 2).mean()) / mean
        assert rel[spp] <= tol, f"{name} {spp} spp: relative RMSE {rel[spp]:.3f} above the stated {tol}"
        assert rel[spp] <= noise, f"{name} {spp} spp: fast-vs-exact {rel[spp]:.3f} exceeds the seed-to-seed noise {noise:.3f}"
        assert abs(lum(fa) / lum(ea) - 1) < ltol, f"{name} {spp} spp: relative luminance off by {lum(fa) / lum(ea) - 1:+.2e}"
    assert rel[256] <= 0.6 * rel[64]                     # Monte-Carlo convergence towards the SAME image (ideal: 0.5)


def test_sample_is_deterministic_and_progressive():
    desc = _desc("cornell", width=120, height=120)
    s = Scene(desc)
    for prec in (EXACT_F64, FAST_F32):
        a = CudaPixelIntegrator(s, precision=prec, seed=9).Sample(4).copy()
        b = CudaPixelIntegrator(s, precision=prec, seed=9).Sample(4).copy()
        assert np.array_equal(a, b)
        c = CudaPixelIntegrator(s, precision=prec, seed=10).Sample(4).copy()
        assert not np.array_equal(a, c)
        lo = CudaPixelIntegrator(s, precision=prec, seed=9).Sample(2, first_sample=0).copy()
        hi = CudaPixelIntegrator(s, precision=prec, seed=9).Sample(2, first_sample=2).copy()
        assert np.allclose((lo + hi)[:, :, :3] / 2, a[:, :, :3], rtol=1e-6, atol=1e-9)


def test_wave_chunking_does_not_change_the_frame(monkeypatch):
    desc = _desc("c1_cube", width=96, height=64)
    ref = {}
    for prec in (EXACT_F64, FAST_F32):
        ref[prec] = CudaPixelIntegrator(Scene(desc), precision=prec, seed=3).Sample(5).copy()
    monkeypatch.setenv("MFX_WAVE_PATHS", "4096")          # < width*height: pixel chunks of one sample each
    monkeypatch.setenv("MFX_WAVE_PATHS_EXACT", "10000")   # 1 sample per wave, 2 pixel chunks ... and uneven tails
    for prec in (EXACT_F64, FAST_F32):
        got = CudaPixelIntegrator(Scene(desc), precision=prec, seed=3).Sample(5).copy()
        if prec == EXACT_F64:
            assert np.array_equal(got, ref[prec])
        else:
            assert np.allclose(got, ref[prec], rtol=1e-5, atol=1e-7)


@pytest.mark.parametrize("world", [2, 3, 8])
def test_tile_sharding_sums_to_the_whole_frame(world):
    desc = _desc("c1_cube", width=200, height=136)
    s = Scene(desc)
    for prec in (EXACT_F64, FAST_F32):
        full = CudaPixelIntegrator(s, precision=prec, seed=2).Sample(3).copy()
        acc = np.zeros_like(full)
        owned = np.zeros(full.shape[:2], int)
        for r in range(world):
            part = CudaPixelIntegrator(s, precision=prec, seed=2, tile_size=32, rank=r, world=world).Sample(3).copy()
            owned += (part[:, :, 3] == 1.0)
            acc += part
        assert (owned == 1).all()
        assert np.array_equal(acc, full)          # RNG keyed on absolute pixel/sample: bit-identical for any world


@pytest.mark.parametrize("world,w,h", [(2, 200, 136), (3, 70, 33), (8, 300, 64), (5, 50, 7), (8, 20, 16)])     # the last: six ranks own nothing
def test_stripe_sharding_assembles_the_whole_frame(world, w, h):
    """Column stripes (MFX_SAMPLE_STRIPES, arithmetic ownership in the kernels -- no pixel table): the ranks' frames are
    disjoint, cover the frame and sum to the one-GPU frame bit for bit; with MFX_SAMPLE_NO_CLEAR a rank touches only its
    own stripes of the output."""
    import torch
    desc = _desc("c1_cube", width=w, height=h)
    s = Scene(desc)
    for prec in (EXACT_F64, FAST_F32):
        full = CudaPixelIntegrator(s, precision=prec, seed=2).Sample(3).copy()
        acc = np.zeros_like(full)
        owned = np.zeros(full.shape[:2], int)
        for r in range(world):
            integ = CudaPixelIntegrator(s, precision=prec, seed=2, tile_size=16, rank=r, world=world)
            part = integ.Sample(3, flags=_lib.SAMPLE_STRIPES).copy()
            own = np.zeros(full.shape[:2], bool)
            own[(np.arange(w) // 16) % world == r, :] = True
            assert np.array_equal(part[:, :, 3] == 1.0, own)
            owned += own
            acc += part
            dev = torch.full((w, h, 4), -7.0, dtype=torch.float64, device="cuda")
            torch.cuda.synchronize()
            integ.SampleDeviceColor(3, dev.data_ptr(), flags=_lib.SAMPLE_STRIPES | _lib.SAMPLE_NO_CLEAR)
            got = dev.cpu().numpy()
            assert np.array_equal(got[own], full[own]) and (got[~own] == -7.0).all()
        assert (owned == 1).all()
        assert np.array_equal(acc, full)


def test_multi_gpu_api_on_the_devices_present():
    """mfx_multi_*: the N-GPU path behind ONE host thread.  With every visible device (1 on the test box, 2..8 under
    gpurun --gpus N) the assembled Color[w,h] and the float frame equal the single-GPU frame bit for bit."""
    from mafrixraytracing_b200 import MultiGpuPixelIntegrator
    n = _lib.load().mfx_device_count()
    for name, kw in (("c1_cube", dict(width=333, height=120)), ("c2_spot", dict(width=480, height=270)), ("cornell", dict(width=24, height=40)),
                     ("random_scene", dict(width=200, height=100))):      # 24 columns: devices beyond the second own nothing; the sphere sample
        desc = _desc(name, **kw)
        single = CudaPixelIntegrator(Scene(desc), precision=FAST_F32, seed=3)
        want = single.Sample(4).copy()
        want32 = single.SampleF32(4)
        for devs in ([0], list(range(n))) if n > 1 else ([0],):
            m = MultiGpuPixelIntegrator(desc, devices=devs, precision=FAST_F32, seed=3)
            assert m.n_devices == len(devs)
            m.Prepare()                                               # layouts uploaded now, not inside the first Sample
            tex = np.full((desc.width, desc.height, 4), -1.0)
            _lib.check(_lib.load().mfx_host_register(_lib.ptr(tex), tex.nbytes))
            try:
                got = m.Sample(4, out=tex)
                assert np.array_equal(got, want)
                tex[:] = -1.0
                m.SampleAsync(4, tex)                                 # the same call without the wait
                with pytest.raises(MafrixError):
                    m.SampleAsync(4, tex)                             # one frame in flight per handle
                m.Wait()
                assert np.array_equal(tex, want)
                m.Wait()                                              # nothing in flight: no-op
            finally:
                _lib.load().mfx_host_unregister(_lib.ptr(tex))
            assert np.array_equal(m.SampleF32(4), want32)                 # pageable destination
            st = m.stats
            assert st["paths"] == desc.width * desc.height * 4 and len(st["per_device"]) == len(devs)
            assert st["closest_rays"] == single.stats["closest_rays"] and st["shadow_rays"] == single.stats["shadow_rays"]
            m.close()
    with pytest.raises(MafrixError):
        MultiGpuPixelIntegrator(_desc("cornell", width=16, height=16), devices=[0, 0])
    with pytest.raises(MafrixError):
        MultiGpuPixelIntegrator(_desc("cornell", width=16, height=16), devices=[n + 3])


def test_cpp_host_drives_several_gpus_through_the_c_abi(tmp_path):
    """host/render_test --gpus N: a single-threaded C++ host (the reference's shape) over mfx_multi_*; its PFM equals
    the one-GPU run's.  Needs >= 2 devices (gpurun --gpus 2); the one-device box checks the refusal instead."""
    import subprocess
    from tests.conftest import ROOT
    exe = os.path.join(ROOT, "host", "render_test")
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "host"), "-s"])
    n = _lib.load().mfx_device_count()
    if n < 2:
        r = subprocess.run([exe, "--gpus", "2", "--frames", "1", "--size", "64x48", "--out", str(tmp_path / "x")], capture_output=True, text=True)
        assert r.returncode == 1 and "device(s) visible" in r.stderr
        return
    a, b = str(tmp_path / "one"), str(tmp_path / "many")
    subprocess.check_call([exe, "--frames", "3", "--spp", "2", "--size", "250x90", "--out", a])
    subprocess.check_call([exe, "--frames", "3", "--spp", "2", "--size", "250x90", "--gpus", str(n), "--out", b])
    assert open(a + ".pfm", "rb").read() == open(b + ".pfm", "rb").read()


def test_async_sample_pipelines_frames_and_equals_the_blocking_call():
    """mfx_pixel_integrator_sample_async / _wait: two frames in flight (frame k downloads while frame k+1 renders), every
    texture equal to the blocking call's, statistics of the frame each wait completes, pageable textures refused."""
    desc = _desc("c2_spot", width=480, height=270)
    s = Scene(desc)
    s.Prepare(FAST_F32)                                                # mfx_scene_prepare: layouts before the first Sample
    integ = CudaPixelIntegrator(s, precision=FAST_F32, seed=4)
    want = [integ.Sample(2, first_sample=2 * k).copy() for k in range(5)]
    rays = integ.stats["closest_rays"]
    lib = _lib.load()
    tex = [np.full((desc.width, desc.height, 4), -1.0) for _ in range(2)]
    with pytest.raises(MafrixError):
        integ.SampleAsync(2, tex[0])                                   # not pinned
    for t in tex:
        _lib.check(lib.mfx_host_register(_lib.ptr(t), t.nbytes))
    try:
        integ.Wait()                                                   # nothing in flight: no-op
        integ.SampleAsync(2, tex[0], first_sample=0)
        for k in range(1, 5):                                          # launch k, then complete k-1
            integ.SampleAsync(2, tex[k % 2], first_sample=2 * k)
            integ.Wait()
            assert np.array_equal(tex[(k - 1) % 2], want[k - 1])
            assert integ.stats["paths"] == desc.width * desc.height * 2
        integ.Wait()
        assert np.array_equal(tex[0], want[4]) and integ.stats["closest_rays"] == rays
        # three launches without a wait: the third completes the first itself; a blocking call drains the rest
        for k in range(3):
            integ.SampleAsync(2, tex[k % 2], first_sample=2 * k)
        assert np.array_equal(integ.Sample(2, first_sample=6), integ.Sample(2, first_sample=6))
        assert np.array_equal(tex[1], want[1]) and np.array_equal(tex[0], want[2])
    finally:
        for t in tex:
            lib.mfx_host_unregister(_lib.ptr(t))
    s.close()


def test_f32_and_device_outputs_agree_with_color_wh():
    import torch
    desc = _desc("cornell", width=90, height=60)
    s = Scene(desc)
    integ = CudaPixelIntegrator(s, precision=FAST_F32, seed=4)
    tex = integ.Sample(3).copy()
    rows = integ.SampleF32(3)
    assert rows.shape == (60, 90, 4)
    assert np.array_equal(rows[:, :, :3], np.transpose(tex[:, :, :3], (1, 0, 2)).astype(np.float32))
    buf = torch.zeros((60, 90, 4), dtype=torch.float32, device="cuda")
    integ.SampleDevice(3, buf.data_ptr())
    torch.cuda.synchronize()
    assert np.array_equal(buf.cpu().numpy(), rows)


# ------------------------------------------------------------------ Film + post-process
def test_film_accumulation_and_tonemap_match_oracle():
    desc = _desc("cornell", width=64, height=48)
    s, o = Scene(desc), oracle.OracleScene(desc)
    integ = CudaPixelIntegrator(s, precision=EXACT_F64, seed=8)
    film = Film(s)
    osum = np.zeros((64, 48, 4))
    for frame in range(3):                       # Scene.Render: GetFrame(pixelIntegrator, 1) per displayed frame
        target = film.GetFrame(integ, 1).copy()
        otarget = oracle.film_add_sample(osum, o.sample(1, seed=8, first_sample=frame), frame + 1.0)
        assert np.array_equal(target[:, :, :3], otarget[:, :, :3])
    assert np.array_equal(film.PostProcess(), oracle.tonemap_rgba8(otarget))
    film.Reset()
    t0 = film.GetFrame(integ, 1, first_sample=0).copy()
    assert np.array_equal(t0[:, :, :3], o.sample(1, seed=8)[:, :, :3])


# ------------------------------------------------------------------ edge cases
def test_degenerate_inputs():
    mats = make_materials([("lambert", (0.7, 0.7, 0.7))])
    light = AreaLight(np.array([(-1, 3, 1), (-1, 3, -1), (1, 3, -1), (1, 3, 1)], float), (0, -1, 0), (10, 10, 10))
    cam = PinholeCamera((0, 1, 4), (0, -0.2, -1), 120.0, 1.0)
    floor = rect_prim((-2, 0, -2), (-2, 0, 2), (2, 0, 2), (2, 0, -2))
    zero_area = make_prims(1)                    # Renault has 4 of these: NaN normal, can never be hit
    zero_area["v"][0, :9] = [0, 1, 0, 0, 1, 0, 1, 1, 0]
    for prims, w, h, depth, spp in [([floor], 1, 1, 0, 1), ([floor], 7, 3, 3, 2), ([floor, zero_area], 16, 16, 2, 2),
                                    ([sphere_prims([(0, 0.5, 0)], 0.5, 0)], 16, 16, 2, 2),
                                    ([floor, sphere_prims([(0, 0.5, 0), (1, 0.3, 0.5)], [0.5, 0.3], 0)], 24, 16, 4, 3)]:
        for mode in (PATH_INTEGRATOR, NEW_PATH_TRACER):
            desc = SceneDesc(np.concatenate(prims), mats, light, cam, w, h, depth, mode)
            s, o = Scene(desc), oracle.OracleScene(desc)
            got = CudaPixelIntegrator(s, precision=EXACT_F64, seed=1).Sample(spp)
            assert np.array_equal(got[:, :, :3], o.sample(spp, seed=1)[:, :, :3])
            fast = CudaPixelIntegrator(s, precision=FAST_F32, seed=1).Sample(spp)
            assert np.isfinite(fast).all()


def test_bad_sample_arguments_raise():
    s = Scene(_desc("cornell", width=16, height=16))
    with pytest.raises(MafrixError):
        CudaPixelIntegrator(s).Sample(0)
    with pytest.raises(MafrixError):
        CudaPixelIntegrator(s, precision=7).Sample(1)
    with pytest.raises(MafrixError):
        CudaPixelIntegrator(s, tile_size=16, rank=2, world=2).Sample(1)
    with pytest.raises(MafrixError):
        CudaPixelIntegrator(s, tile_size=0, rank=0, world=2).Sample(1)


def test_supplied_tree_is_used_and_equals_host_build():
    desc = _desc("c2_spot", width=64, height=36)
    b = Bvh.Build(desc.prims)
    s1, s2 = Scene(desc), Scene(desc, bvh=b)
    got = s2.bvh()
    assert np.array_equal(got.indices, b.indices) and np.array_equal(got.nodes.view(np.uint8), b.nodes.view(np.uint8))
    a = CudaPixelIntegrator(s1, precision=EXACT_F64, seed=1).Sample(1).copy()
    c = CudaPixelIntegrator(s2, precision=EXACT_F64, seed=1).Sample(1).copy()
    assert np.array_equal(a, c)


# ------------------------------------------------------------------ full-size properties (BASELINE configs[1])
def test_c2_full_size_properties():
    desc = scenes.c2_spot()
    s = Scene(desc)
    integ = CudaPixelIntegrator(s, precision=FAST_F32, seed=1)
    a = integ.SampleF32(2)
    st = dict(integ.stats)
    assert st["paths"] == 1920 * 1080 * 2
    assert st["paths"] <= st["closest_rays"] <= st["paths"] * (desc.max_depth + 1)
    assert st["shadow_rays"] <= st["closest_rays"]
    b = integ.SampleF32(2)
    assert np.array_equal(a, b)                                   # idempotent / deterministic
    acc = np.zeros_like(a)
    for r in range(8):                                            # 8-way interleaved 64x64 tiles
        acc += CudaPixelIntegrator(s, precision=FAST_F32, seed=1, tile_size=64, rank=r, world=8).SampleF32(2)
    assert np.array_equal(acc, a)
    # the exact frame of the same samples (matched random stream): f32 frame within the stated tolerance at full size
    m = integ.SampleF32(2, flags=_lib.SAMPLE_REFERENCE_STREAM)
    e = np.transpose(CudaPixelIntegrator(s, precision=EXACT_F64, seed=1).Sample(2)[:, :, :3], (1, 0, 2))
    rel = np.sqrt(((m[:, :, :3] - e) ** 2).mean()) / np.abs(e).mean()
    assert rel < 5e-2
    # the production sampler estimates the same frame: means agree (2 spp of 2 M pixels)
    assert abs(a[:, :, :3].mean() / e.mean() - 1) < 5e-3


def test_traversal_counters_match_oracle_ordered_counts():
    desc = _desc("c2_spot", width=192, height=108)
    s, o = Scene(desc), oracle.OracleScene(desc)
    integ = CudaPixelIntegrator(s, precision=FAST_F32, seed=2)
    integ.Sample(2, flags=_lib.SAMPLE_COUNT_TRAVERSAL)
    st = integ.stats
    _, ost = o.sample(2, seed=2, stats=True, count_ordered=True)
    for c, rays in ((0, st["closest_rays"]), (1, st["shadow_rays"])):
        g_nodes, g_tris = st["nodes"][c] / rays, st["tris"][c] / rays
        o_nodes, o_tris = ost["ord_nodes"][c] / ost["ord_rays"][c], ost["ord_tris"][c] / ost["ord_rays"][c]
        assert abs(g_nodes / o_nodes - 1) < 0.10 and abs(g_tris / o_tris - 1) < 0.10, (c, g_nodes, o_nodes, g_tris, o_tris)


def test_own_tree_counters_and_image_match_the_reference_tree_run():
    """MFX_SAMPLE_COUNT_OWN_TREE instruments the shipped kernel on the library's SAH tree: it must fetch far fewer
    records than the reference tree has node tests, and render the same frame as the uninstrumented run.  The
    reference-tree run (k_f_trace4) must render that frame too: a nearest-hit query has one answer whichever tree finds
    it, so only pixels behind one of the rare tie-broken hits may change."""
    desc = _desc("c2_spot", width=240, height=135)
    s = Scene(desc)
    integ = CudaPixelIntegrator(s, precision=FAST_F32, seed=2)
    plain = integ.Sample(2, flags=_lib.SAMPLE_F32_PRIMARY).copy()      # the instrumented kernel is the f32 one, bounce 0 included
    own = integ.Sample(2, flags=_lib.SAMPLE_COUNT_OWN_TREE).copy()
    so = dict(integ.stats)
    assert np.array_equal(plain, own)
    ref = integ.Sample(2, flags=_lib.SAMPLE_COUNT_TRAVERSAL).copy()
    sr = dict(integ.stats)
    assert (plain != ref).any(axis=2).mean() <= 5e-3
    assert so["closest_rays"] == sr["closest_rays"] or abs(so["closest_rays"] / sr["closest_rays"] - 1) < 1e-3
    for c, rays in ((0, "closest_rays"), (1, "shadow_rays")):
        rec, ref_nodes = so["nodes"][c] / so[rays], sr["nodes"][c] / sr[rays]
        assert 1.0 <= rec < 0.25 * ref_nodes, (c, rec, ref_nodes)          # 128 B records vs 32 B reference nodes
        assert so["tris"][c] / so[rays] < sr["tris"][c] / sr[rays]


def test_wave_grows_with_the_call_and_frames_do_not_depend_on_it():
    """The path-state wave is sized for pixels x spp of the call and only grows: a scene that first renders 1 spp and
    then 40 spp must give the same 40-spp frame as a fresh scene (and as a run chunked into small waves)."""
    desc = _desc("c1_cube", width=320, height=200)
    a = Scene(desc)
    ia = CudaPixelIntegrator(a, precision=FAST_F32, seed=6)
    ia.Sample(1)
    grown = ia.Sample(40).copy()
    fresh = CudaPixelIntegrator(Scene(desc), precision=FAST_F32, seed=6).Sample(40).copy()
    assert np.array_equal(grown, fresh)
    p, t = a.TracePrimary(np.random.default_rng(0).random((300000, 2)), precision=FAST_F32)     # seam after growth
    assert (p >= 0).all() and np.isfinite(t).all()


@pytest.mark.parametrize("name,width,height,spp", [("cornell", 50, 37, 6), ("c1_cube", 97, 33, 5), ("c2_spot", 200, 112, 48), ("spheres", 64, 48, 16)])
def test_frames_do_not_depend_on_the_order_of_the_path_ids(monkeypatch, name, width, height, spp):
    """Path ids walk the frame in 8-pixel column stripes with blocks of 16 samples of a pixel next to each other
    (path_split / pixel_of: coherence for the warps, DESIGN.md 3).  The RNG is keyed on pixel and sample, so the frame
    must be the one the row-major, sample-major order of round 1 gives -- for widths that are no multiple of the stripe,
    sample counts that are no multiple of the block, and frames cut into several waves of pixels or of samples."""
    desc = _desc(name, width=width, height=height)
    s = Scene(desc)
    integ = CudaPixelIntegrator(s, precision=FAST_F32, seed=9)
    monkeypatch.setenv("MFX_PIXEL_STRIPE", "0"); monkeypatch.setenv("MFX_SAMPLE_BLOCK_LOG2", "0")
    ref = integ.Sample(spp).copy()
    rays = integ.stats["closest_rays"] + integ.stats["shadow_rays"]
    for stripe, blk, wave in (("8", "4", None), ("4", "6", None), ("16", "2", None), ("8", "4", str(width * height * 2 + 7)), ("8", "4", str(width * 3))):
        monkeypatch.setenv("MFX_PIXEL_STRIPE", stripe); monkeypatch.setenv("MFX_SAMPLE_BLOCK_LOG2", blk)
        if wave:
            monkeypatch.setenv("MFX_WAVE_PATHS", wave)
        sc = Scene(desc)                                     # a fresh scene: the wave is sized under the new cap
        it = CudaPixelIntegrator(sc, precision=FAST_F32, seed=9)
        img = it.Sample(spp).copy()
        assert np.array_equal(img, ref), (stripe, blk, wave)
        assert it.stats["closest_rays"] + it.stats["shadow_rays"] == rays
        sc.close()
        monkeypatch.delenv("MFX_WAVE_PATHS", raising=False)


def test_wave_shrinks_when_the_gpu_is_nearly_full():
    """Another tenant holds almost all HBM: the path-state wave (6.5 GB wanted here) must fall back to a smaller one
    -- more launches, same frame -- instead of failing."""
    import torch
    desc = _desc("c2_spot", width=1920, height=1080)
    spp = 17                                        # 35 M paths x 184 B = 6.5 GB of path state, a size no other test leaves pooled
    torch.cuda.synchronize()
    free, _total = torch.cuda.mem_get_info()
    hog = torch.empty(max(free - (3 << 30), 1 << 20), dtype=torch.uint8, device="cuda")
    try:
        got = CudaPixelIntegrator(Scene(desc), precision=FAST_F32, seed=3).SampleF32(spp)
    finally:
        del hog
        torch.cuda.empty_cache()
    want = CudaPixelIntegrator(Scene(desc), precision=FAST_F32, seed=3).SampleF32(spp)
    assert np.allclose(got, want, rtol=1e-5, atol=1e-7)


def tiny_tree_scene(n_tris):
    """n_tris random triangles on a 3-wide grid: one to nine of them give a one-record tree with 1..4 leaves (a
    single-leaf root, empty links) or the first two-level trees."""
    rng = np.random.default_rng(n_tris)
    prims = make_prims(n_tris)
    for i in range(n_tris):
        c = np.array([(i % 3) - 1.0, (i // 3) - 1.0, -0.3 * i])
        prims["v"][i, :9] = (c + rng.uniform(-0.45, 0.45, (3, 3))).ravel()
    mats = make_materials([("lambert", (0.7, 0.7, 0.7))])
    light = AreaLight(np.array([(-1, 3, 1), (-1, 3, -1), (1, 3, -1), (1, 3, 1)], float), (0, -1, 0), (10, 10, 10))
    cam = PinholeCamera((0, 0, 4), (0, 0, -1), 120.0, 1.0)
    return SceneDesc(prims, mats, light, cam, 64, 64, 2, PATH_INTEGRATOR)


@pytest.mark.parametrize("n_tris", [1, 2, 3, 5, 9])
def test_tiny_own_trees(n_tris):
    """One-record trees with 1..4 leaves and the first two-level trees: fast ids must equal the oracle's."""
    rng = np.random.default_rng(n_tris)
    rng.uniform(-0.45, 0.45, (n_tris, 3, 3))                # the draws tiny_tree_scene made: the same rays as before
    desc = tiny_tree_scene(n_tris)
    s, o = Scene(desc), oracle.OracleScene(desc)
    uv = rng.random((20000, 2))
    op, ot = o.trace_primary(uv)
    fp, ft = s.TracePrimary(uv, precision=FAST_F32)
    assert np.array_equal(fp, op) and np.array_equal(ft, ot)
    assert np.isfinite(CudaPixelIntegrator(s, precision=FAST_F32, seed=1).Sample(2)).all()


def test_coincident_primitives_and_deepest_paths():
    """200 copies of one triangle (no centroid spread: the own-tree builder must still terminate and balance) in front
    of a floor, traced with the deepest path length the library allows (max_depth 15 = 16 vertices)."""
    tri = make_prims(200)
    tri["v"][:, :9] = [-0.5, 0.2, 0.0, 0.5, 0.2, 0.0, 0.0, 1.2, 0.0]
    floor = rect_prim((-3, 0, -3), (-3, 0, 3), (3, 0, 3), (3, 0, -3))
    mats = make_materials([("lambert", (0.8, 0.8, 0.8))])
    light = AreaLight(np.array([(-1, 3, 1), (-1, 3, -1), (1, 3, -1), (1, 3, 1)], float), (0, -1, 0), (10, 10, 10))
    cam = PinholeCamera((0, 1, 4), (0, -0.1, -1), 120.0, 1.0)
    desc = SceneDesc(np.concatenate([tri, floor]), mats, light, cam, 64, 64, 15, PATH_INTEGRATOR)
    s, o = Scene(desc), oracle.OracleScene(desc)
    uv = np.random.default_rng(3).random((20000, 2))
    op, ot = o.trace_primary(uv)
    fp, ft = s.TracePrimary(uv, precision=FAST_F32)
    hit_tri = (op >= 0) & (op < 200)
    assert hit_tri.sum() > 100
    assert np.array_equal(fp, op) and np.array_equal(ft, ot)          # 200-way exact ties: the reference's tie rule decides
    exact = CudaPixelIntegrator(s, precision=EXACT_F64, seed=2).Sample(2)
    assert np.array_equal(exact[:, :, :3], o.sample(2, seed=2)[:, :, :3])
    fast = CudaPixelIntegrator(s, precision=FAST_F32, seed=2).Sample(8)
    assert np.isfinite(fast).all() and fast[:, :, :3].mean() > 0


def test_ingested_xml_scene_renders_like_the_procedural_one(tmp_path):
    """Scene.xml-style description + OBJ (mafrixraytracing_b200/ingest.py) -> same frame, bit for bit, as the
    procedural Cornell scene; the oracle agrees."""
    from tests.test_ingest import _write_cornell
    from mafrixraytracing_b200.ingest import init_scene_state
    xml, want = _write_cornell(str(tmp_path))
    desc = init_scene_state(xml, base_dir=str(tmp_path))
    desc.width = want.width = 120
    desc.height = want.height = 120
    a = CudaPixelIntegrator(Scene(desc), precision=EXACT_F64, seed=4).Sample(2).copy()
    b = CudaPixelIntegrator(Scene(want), precision=EXACT_F64, seed=4).Sample(2).copy()
    assert np.array_equal(a, b)
    assert np.array_equal(a[:, :, :3], oracle.OracleScene(desc).sample(2, seed=4)[:, :, :3])
    f = CudaPixelIntegrator(Scene(desc), precision=FAST_F32, seed=4).Sample(2).copy()
    g = CudaPixelIntegrator(Scene(want), precision=FAST_F32, seed=4).Sample(2).copy()
    assert np.array_equal(f, g)


def test_headless_render_cli_from_a_scene_file(tmp_path):
    """python -m mafrixraytracing_b200.render scene.xml: the RenderTest loop without the window."""
    from tests.test_ingest import _write_cornell
    from mafrixraytracing_b200 import render
    xml, want = _write_cornell(str(tmp_path))
    (tmp_path / "scene.xml").write_text(xml.replace('value="300"', 'value="96"'))
    out = str(tmp_path / "img")
    assert render.main([str(tmp_path / "scene.xml"), "--frames", "3", "--spp", "2", "--out", out]) == 0
    with open(out + ".pfm", "rb") as fh:
        assert fh.readline() == b"PF\n" and fh.readline() == b"96 96\n" and fh.readline() == b"-1.0\n"
        img = np.frombuffer(fh.read(), "<f4").reshape(96, 96, 3)[::-1]
    want.width = want.height = 96
    s = Scene(want)
    film = Film(s)
    integ = CudaPixelIntegrator(s, precision=FAST_F32, seed=1)
    for f in range(3):
        target = film.GetFrame(integ, 2, first_sample=2 * f)
    assert np.array_equal(img, np.transpose(target[:, :, :3], (1, 0, 2)).astype(np.float32))
    png = open(out + ".png", "rb").read()
    assert png[:8] == b"\x89PNG\r\n\x1a\n" and png[12:16] == b"IHDR" and png[16:24] == (96).to_bytes(4, "big") * 2
    import zlib
    idat = png[png.index(b"IDAT") + 4: png.index(b"IEND") - 8]
    rows = np.frombuffer(zlib.decompress(idat), np.uint8).reshape(96, 1 + 96 * 4)[:, 1:].reshape(96, 96, 4)
    assert np.array_equal(rows, film.PostProcess())


def test_cpp_host_driver_matches_python_host(tmp_path):
    """host/render_test (the C++ mirror of RenderTest/RayTracing4.fs) against the ctypes host: same
    Film loop, same frames -> same PFM."""
    import subprocess
    from tests.conftest import ROOT
    exe = os.path.join(ROOT, "host", "render_test")
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "host"), "-s"])
    out = str(tmp_path / "cornell")
    subprocess.check_call([exe, "--frames", "3", "--spp", "2", "--size", "120x90", "--out", out])
    with open(out + ".pfm", "rb") as fh:
        assert fh.readline() == b"PF\n" and fh.readline() == b"120 90\n" and fh.readline() == b"-1.0\n"
        img = np.frombuffer(fh.read(), "<f4").reshape(90, 120, 3)[::-1]
    s = Scene(scenes.cornell(width=120, height=90))
    film = Film(s)
    integ = CudaPixelIntegrator(s, precision=FAST_F32, seed=1)
    for f in range(3):
        target = film.GetFrame(integ, 2, first_sample=2 * f)
    want = np.transpose(target[:, :, :3], (1, 0, 2)).astype(np.float32)
    assert np.array_equal(img, want)


def test_film_checkpoint_resume_is_exact():
    desc = _desc("cornell", width=48, height=40)
    s = Scene(desc)
    integ = CudaPixelIntegrator(s, precision=EXACT_F64, seed=5)
    a = Film(s)
    for _ in range(4):
        full = a.GetFrame(integ, 2).copy()
    b = Film(s)
    for _ in range(2):
        b.GetFrame(integ, 2)
    saved, count = b.Export()
    assert count == 2.0
    c = Film(Scene(desc))                      # a fresh process would do exactly this
    c.Import(saved, count)
    integ2 = CudaPixelIntegrator(c.scene, precision=EXACT_F64, seed=5)
    for _ in range(2):
        resumed = c.GetFrame(integ2, 2).copy()   # first_sample continues at frameCount * spp
    assert np.array_equal(resumed, full)
    assert np.array_equal(c.PostProcess(), a.PostProcess())
