"""Path-by-path parity of the fast f32 renderer against the f64 reference, per material and bounce depth.

Bounce 0 of a fast frame is pinned bit for bit elsewhere (test_gpu_parity.py).  Everything after it -- the f32
primitive tests of k_f_trace6 for closest hits from surfaces and for every shadow query, the f32 BSDF, light and
throughput arithmetic of k_f_shade, and k_f_shade_sky / sky_scatter_f of the sky tracer -- is checked here against the
f64 renderer in two ways.

1. Matched stream.  A 1-spp frame with MFX_SAMPLE_REFERENCE_STREAM runs the reference's rejection samplers on the exact
   mode's Philox stream, so every pixel holds ONE path and the f64 renderer (the oracle, and EXACT_F64, which must equal
   it bit for bit) computes the same path.  Per path, r = max over RGB |f - e| / max(max |e|, floor), the floor being
   FLOOR_FRAC of the mean radiance of the case.  A path with r > TAU took another decision in f32 (another hit, the
   other side of an occluder edge, a flipped total internal reflection): the share of such paths, and their share of
   the radiance, are bounded per case.  The agreeing paths must be accurate (median and 99.9th percentile of r) and
   unbiased (signed mean relative error), which is what catches a wrong constant or a missing normalisation.

2. Default sampler.  The production sampler (uniform_hemisphere_f, the metal radius from spare bits, the coin from a
   low bit, the sky's ball point) draws from its own stream, so it is compared in expectation: B independent batches in
   FAST_F32 and in EXACT_F64, each batch's mean over the frame and over each tile of a 4x4 grid taken as one sample,
   two-sample z-scores bounded.  Each case carries enough paths that a 1 % change of the frame is at least 8 standard
   errors (asserted, not assumed).

Bars were set from a B200 run: each carries the value measured there and sits at about twice it."""
import numpy as np
import pytest

from mafrixraytracing_b200 import scenes, Scene, CudaPixelIntegrator, EXACT_F64, FAST_F32, _lib
from mafrixraytracing_b200.scene import (AreaLight, PinholeCamera, RayTraceCamera, SceneDesc, make_materials,
                                         sphere_prims, NEW_PATH_TRACER, PATH_INTEGRATOR)
from oracle import oracle
from .test_gpu_traversal_stack import _haystack
from .test_oracle_sky import sky_desc

pytestmark = pytest.mark.gpu

TAU = 1e-3              # a path whose relative difference exceeds this took another decision in f32
FLOOR_FRAC = 1e-2       # r's denominator never drops below this fraction of the case's mean radiance


# ------------------------------------------------------------------ scenes
def material_scene(spec, integrator=NEW_PATH_TRACER, width=320, height=200, max_depth=4):
    """A floor, a planar back Rect, four small spheres (the f32 residual-form roots) and one sphere of radius 40 behind
    them (the kernels' f64 big-sphere branch), every surface of the one material `spec` (make_materials form), under a
    2x2 area light."""
    floor = scenes.quad_facing((-8, 0, -8), (-8, 0, 8), (8, 0, 8), (8, 0, -8), (0, 1, 0), 0)
    wall = scenes.quad_facing((-2.5, 0, -2.2), (2.5, 0, -2.2), (2.5, 2.4, -2.2), (-2.5, 2.4, -2.2), (0, 0, 1), 0)
    small = sphere_prims([(-1.3, 0.45, 0.2), (0.0, 0.6, 0.7), (1.2, 0.35, -0.3), (0.5, 1.5, -1.2)], [0.45, 0.6, 0.35, 0.3], 0)
    big = sphere_prims([(0.0, 2.0, -46.0)], 40.0, 0)
    light = AreaLight(np.array([(-1, 4, 1), (-1, 4, -1), (1, 4, -1), (1, 4, 1)], float), (0, -1, 0), (10, 10, 10))
    cam = PinholeCamera((0, 1.6, 5), (0, -0.25, -1), 120.0, width / height)
    return SceneDesc(np.concatenate([floor, wall, small, big]), make_materials([spec]), light, cam, width, height,
                     max_depth, integrator, name=spec[0])


def sky_material_scene(spec, width=320, height=200, max_depth=50):
    """The sky tracer's scene for one material: the r = 1000 ground sphere and four spheres on it, all of `spec`."""
    rf, pm = scenes.perlin_tables(5)
    cam = RayTraceCamera((0.5, 1.8, 6.0), (0, 0.5, 0), (0, 1, 0), 40.0, width / height)
    return sky_desc([(0, -1000, 0), (-1.6, 0.7, 0), (0, 1, -0.5), (1.5, 0.5, 0.6), (0.6, 0.3, 2.0)],
                    [1000, 0.7, 1.0, 0.5, 0.3], [spec] * 5, width=width, height=height, max_depth=max_depth, cam=cam,
                    tables=(rf, pm))


MATERIALS = {
    "lambert": ("lambert", (0.7, 0.6, 0.5)),
    "metal0": ("metal", (0.8, 0.7, 0.6), 0.0),
    "metal0.3": ("metal", (0.8, 0.7, 0.6), 0.3),
    "metal1": ("metal", (0.8, 0.7, 0.6), 1.0),
    "metal1.7": ("metal", (0.8, 0.7, 0.6), 1.7),            # min(fuzz, 1) caps it
    "glass_in": ("spectrans", (1.0, 1.0, 1.0), 1.0, 1.5),
    "glass_out": ("spectrans", (1.0, 1.0, 1.0), 1.5, 1.0),  # rays leave the spheres from inside; total internal reflection
}
SKY_MATERIALS = {
    "constant": ("lambert", (0.7, 0.6, 0.5)),
    "checker": ("checker", (0.2, 0.3, 0.1), (0.9, 0.9, 0.9)),
    "noise": ("noise",),
    "metal": ("metal", (0.8, 0.7, 0.6), 0.3),
    "dielectric": ("dielectric", 1.5),
}


def build_case(name, depth):
    """(desc, frames): frames 1-spp frames of the case make about 1e6 paths."""
    if name in ("cornell", "c1_cube"):
        return scenes.WORKLOADS[name](width=320, height=320, max_depth=depth), 10
    if name in ("c2_spot", "c3_renault"):
        return scenes.WORKLOADS[name](width=320, height=180, max_depth=depth), 17
    if name == "haystack":
        return _haystack(width=320, height=180, max_depth=depth), 17
    if name.startswith("sky_"):
        return sky_material_scene(SKY_MATERIALS[name[4:]], max_depth=depth), 16
    if name == "A_glass":
        return material_scene(MATERIALS["glass_in"], integrator=PATH_INTEGRATOR, max_depth=depth), 16
    return material_scene(MATERIALS[name], max_depth=depth), 16


# ------------------------------------------------------------------ matched-stream paths
def render_paths(desc, frames, seed=3, oracle_frames=None):
    """(fast, exact) radiance of frames x width x height single paths, (n, 3) each.  The exact side is EXACT_F64, and
    its first `oracle_frames` frames (default: all) must equal the CPU oracle's bit for bit."""
    s = Scene(desc)
    o = oracle.OracleSkyScene(desc) if desc.sky is not None else oracle.OracleScene(desc)
    fast = CudaPixelIntegrator(s, precision=FAST_F32, seed=seed)
    exact = CudaPixelIntegrator(s, precision=EXACT_F64, seed=seed)
    f, e = [], []
    for k in range(frames):
        got = exact.Sample(1, first_sample=k)[:, :, :3].copy()
        if oracle_frames is None or k < oracle_frames:
            assert np.array_equal(got, o.sample(1, seed=seed, first_sample=k)[:, :, :3]), f"EXACT_F64 frame {k} differs from the oracle"
        e.append(got.reshape(-1, 3))
        f.append(fast.Sample(1, first_sample=k, flags=_lib.SAMPLE_REFERENCE_STREAM)[:, :, :3].reshape(-1, 3).copy())
    s.close()
    return np.concatenate(f), np.concatenate(e)


def path_stats(f, e):
    """The per-path measures of the module docstring, as one dict."""
    floor = FLOOR_FRAC * np.abs(e).max(axis=1).mean()
    den = np.maximum(np.abs(e).max(axis=1), floor)
    r = np.abs(f - e).max(axis=1) / den
    agree = r <= TAU
    fs, es = f.sum(axis=1), e.sum(axis=1)
    lit = agree & (es > floor)
    return dict(
        paths=len(r),
        diverged=float((~agree).mean()),
        median=float(np.median(r[agree])) if agree.any() else np.inf,
        p999=float(np.percentile(r[agree], 99.9)) if agree.any() else np.inf,
        bias=float(((fs[lit] - es[lit]) / es[lit]).mean()) if lit.any() else np.inf,
        diverged_mass=float(np.abs(f[~agree] - e[~agree]).sum() / max(np.abs(e).sum(), 1e-300)),
        finite=bool(np.isfinite(f).all()),
        negative=int(((f < 0) & (e >= 0)).any(axis=1).sum()),
        negative_agreeing=int((((f < 0) & (e >= 0)).any(axis=1) & agree).sum()),
        black=float(((fs == 0) & (es != 0)).mean()),
    )


# ------------------------------------------------------------------ default sampler in expectation
def batch_means(render, batches, spp, width, height, clip=None):
    """(batches, 17): per batch, the mean radiance (RGB summed, optionally clipped per pixel at `clip`) over the frame,
    then over each tile of a 4x4 grid.  render(spp, first_sample) -> (width, height, >=3) frame."""
    out = np.zeros((batches, 17))
    xs = np.linspace(0, width, 5).astype(int)
    ys = np.linspace(0, height, 5).astype(int)
    for b in range(batches):
        img = render(spp, b * spp)[:, :, :3].sum(axis=2)
        if clip is not None:
            img = np.minimum(img, clip)
        out[b, 0] = img.mean()
        out[b, 1:] = [img[xs[i]:xs[i + 1], ys[j]:ys[j + 1]].mean() for i in range(4) for j in range(4)]
    return out


def z_scores(a, b):
    """Two-sample z of the batch means: (frame z, worst tile |z|, relative standard error of the frame difference)."""
    se = np.sqrt(a.var(axis=0, ddof=1) / len(a) + b.var(axis=0, ddof=1) / len(b))
    diff = a.mean(axis=0) - b.mean(axis=0)
    # a tile that is black in every batch of both renderers agrees exactly
    z = np.where(se > 0, diff / np.where(se > 0, se, 1.0), np.where(diff == 0, 0.0, np.inf))
    return float(z[0]), float(np.abs(z[1:]).max()), float(se[0] / abs(b[:, 0].mean()))


# ------------------------------------------------------------------ 1. matched stream, path by path
# Global bars on the agreeing paths (worst case measured on a B200 in brackets):
MEDIAN_BAR = 5e-7       # median r                                        [2.2e-7, c1_cube depth 3]
P999_BAR = 8e-5         # 99.9th percentile of r                          [4.0e-5, sky_metal depth 50]
BIAS_BAR = 1.5e-6       # |signed mean of (f - e) / e|                    [5.4e-7, haystack depth 0]

# Per case: share of diverged paths and their share of the radiance, each bar with the value measured on a B200.
# Each bar is about twice the measured value and at least the measured value plus five paths.
#           (scene, max_depth): (diverged bar, measured, diverged-mass bar, measured)
CASES = {
    ("cornell", 0): (5.9e-06, 9.8e-07, 5.1e-06, 2.1e-10),
    ("cornell", 1): (0.00059, 0.00029, 6.1e-06, 1.1e-06),
    ("cornell", 3): (0.0011, 0.00053, 6.9e-06, 1.9e-06),
    ("c1_cube", 0): (4.9e-06, 0, 5e-06, 0),
    ("c1_cube", 1): (5.9e-06, 9.8e-07, 5.1e-06, 7.9e-12),
    ("c1_cube", 3): (6.9e-06, 2e-06, 5.1e-06, 4.7e-11),
    ("c2_spot", 5): (1.1e-05, 5.1e-06, 8.1e-06, 3e-06),
    ("haystack", 0): (1.1e-05, 5.1e-06, 4.3e-05, 2.1e-05),
    ("haystack", 2): (0.00018, 8.6e-05, 0.0005, 0.00025),
    ("lambert", 0): (4.9e-06, 0, 5e-06, 0),
    ("lambert", 1): (4.9e-06, 0, 5e-06, 0),
    ("lambert", 4): (4.9e-06, 0, 5e-06, 0),
    ("metal0", 0): (4.9e-06, 0, 5e-06, 0),
    ("metal0", 1): (5.9e-06, 9.8e-07, 5.1e-06, 9.2e-12),
    ("metal0", 4): (1.4e-05, 6.8e-06, 5.1e-06, 6.2e-10),
    ("metal0.3", 0): (4.9e-06, 0, 5e-06, 0),
    ("metal0.3", 1): (5.9e-06, 9.8e-07, 5.1e-06, 7e-08),
    ("metal0.3", 4): (1.6e-05, 7.8e-06, 5.1e-06, 6.9e-08),
    ("metal1", 0): (4.9e-06, 0, 5e-06, 0),
    ("metal1", 1): (4.9e-06, 0, 5e-06, 0),
    ("metal1", 4): (6.9e-06, 2e-06, 5.1e-06, 3e-09),
    ("metal1.7", 0): (4.9e-06, 0, 5e-06, 0),
    ("metal1.7", 1): (4.9e-06, 0, 5e-06, 0),
    ("metal1.7", 4): (6.9e-06, 2e-06, 5.1e-06, 3e-09),
    ("glass_in", 0): (4.9e-06, 0, 5e-06, 0),
    ("glass_in", 1): (9.8e-06, 4.9e-06, 5.1e-06, 7.3e-10),
    ("glass_in", 4): (1.6e-05, 7.8e-06, 5.1e-06, 4.2e-09),
    ("glass_out", 0): (4.9e-06, 0, 5e-06, 0),
    ("glass_out", 1): (9.8e-06, 4.9e-06, 5.1e-06, 4.3e-09),
    ("glass_out", 4): (8.8e-06, 3.9e-06, 5.1e-06, 4.2e-09),
    ("c3_renault", 5): (0.00086, 0.00043, 0.0028, 0.0014),
    ("sky_constant", 2): (4.9e-06, 0, 5e-06, 0),
    ("sky_constant", 50): (2.2e-05, 1.1e-05, 5.2e-06, 1.7e-07),
    ("sky_checker", 2): (8.8e-06, 3.9e-06, 8.2e-06, 3.2e-06),
    ("sky_checker", 50): (4.5e-05, 2.2e-05, 8.5e-06, 3.5e-06),
    ("sky_noise", 2): (5.9e-06, 9.8e-07, 5.8e-06, 7.4e-07),
    ("sky_noise", 50): (3e-05, 1.5e-05, 6.2e-06, 1.1e-06),
    ("sky_metal", 2): (5.9e-06, 9.8e-07, 5.8e-06, 7.1e-07),
    ("sky_metal", 50): (0.00023, 0.00011, 5.3e-06, 2.4e-07),
    ("sky_dielectric", 2): (4.9e-06, 0, 5e-06, 0),
    ("sky_dielectric", 50): (4.9e-06, 0, 5e-06, 0),
}


@pytest.mark.parametrize("name,depth", list(CASES))
def test_fast_paths_track_the_f64_paths(name, depth):
    """One path per pixel on the matched stream, compared with the same path in f64.  Depth 0 is raygen, the id-exact
    bounce 0, shade b0 and one f32 shadow query with a per-ray distance; each further bounce adds k_f_trace6 closest
    hits from surface origins with the source primitive excluded."""
    div_bar, div_meas, mass_bar, mass_meas = CASES[(name, depth)]
    desc, frames = build_case(name, depth)
    # the haystack's reference tree is slow on the CPU: its oracle checks two of the 17 EXACT_F64 frames
    f, e = render_paths(desc, frames, oracle_frames=2 if name == "haystack" else None)
    st = path_stats(f, e)
    msg = f"{name} depth {depth}: {st}"
    assert st["finite"], msg                                                            # (e)
    # a channel the f64 path leaves >= 0 goes negative only on a path that took another decision (PathIntegrator lights
    # the back of a surface with negative radiance, and the haystack, Cornell and C3 show such paths), and never in
    # the single-material scenes
    assert st["negative_agreeing"] == 0, msg
    if name in MATERIALS or name.startswith("sky_"):
        assert st["negative"] == 0, msg
    assert st["diverged"] <= div_bar, msg                                               # (a)
    assert st["median"] <= MEDIAN_BAR and st["p999"] <= P999_BAR, msg                   # (b)
    assert abs(st["bias"]) <= BIAS_BAR, msg                                             # (c)
    assert st["diverged_mass"] <= mass_bar, msg                                         # (d)


def test_mode_a_specular_transmission_is_black_past_its_vertex():
    """PathIntegrator gives SpecularTransmission no BSDF value (z = 0 in k_f_shade): a path ends black at such a vertex,
    light sample included.  Every surface of this scene is of that material, so every frame is exactly black in both
    samplers of the fast path, as in the f64 renderer."""
    desc, _ = build_case("A_glass", 3)
    s = Scene(desc)
    assert not CudaPixelIntegrator(s, precision=EXACT_F64, seed=3).Sample(4)[:, :, :3].any()
    for flags in (0, _lib.SAMPLE_REFERENCE_STREAM):
        img = CudaPixelIntegrator(s, precision=FAST_F32, seed=3).Sample(4, flags=flags)
        assert not img[:, :, :3].any(), flags
    s.close()


# ------------------------------------------------------------------ 2. the default sampler in expectation
BATCHES, SPP = 32, 4
Z_FRAME, Z_TILE = 5.0, 5.5
SPECTRANS_CLIP = 100.0   # per-pixel clip of the heavy-tailed 1/|cos| scenes, the same for both renderers


def default_sampler_scene(name):
    if name == "lambert_A":
        return material_scene(MATERIALS["lambert"], integrator=PATH_INTEGRATOR)
    if name.startswith("sky_"):
        return sky_material_scene(SKY_MATERIALS[name[4:]])
    return material_scene(MATERIALS[name])


@pytest.mark.parametrize("name", ["lambert_A"] + list(MATERIALS) + ["sky_" + m for m in SKY_MATERIALS])
def test_default_sampler_has_the_reference_expectation(name):
    """FAST_F32 with its default sampler against EXACT_F64, BATCHES independent batches each (distinct first_sample
    ranges, different seeds): the frame mean and the 16 tile means must agree within the z bars, and the batches must
    carry enough paths that a 1 % change of the frame is at least 8 standard errors."""
    desc = default_sampler_scene(name)
    s = Scene(desc)
    clip = SPECTRANS_CLIP if name.startswith("glass") else None
    fi = CudaPixelIntegrator(s, precision=FAST_F32, seed=21)
    ei = CudaPixelIntegrator(s, precision=EXACT_F64, seed=22)
    fa = batch_means(lambda n, k: fi.Sample(n, first_sample=k), BATCHES, SPP, desc.width, desc.height, clip)
    ea = batch_means(lambda n, k: ei.Sample(n, first_sample=k), BATCHES, SPP, desc.width, desc.height, clip)
    s.close()
    z, zt, se = z_scores(fa, ea)
    assert 8 * se <= 0.01, f"{name}: relative standard error {se:.2e} is too large to see a 1 % change"
    assert abs(z) <= Z_FRAME and zt <= Z_TILE, f"{name}: frame z {z:+.2f}, worst tile |z| {zt:.2f}"
