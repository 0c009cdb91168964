"""Small end-to-end run for compute-sanitizer: every fast/exact/hybrid kernel, all three integrators, spheres incl. the f64
big one, own-tree and reference-tree counters, Film + tone map / sky display, seams (id-exact and f32, incl. the
exact fixup of axis-parallel rays), tiles and stripes, the async entry point, mfx_multi_* on the visible devices."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
from mafrixraytracing_b200 import scenes, Scene, CudaPixelIntegrator, MultiGpuPixelIntegrator, Film, EXACT_F64, FAST_F32, _lib
for name, kw in [("cornell", dict(width=64, height=48)), ("c2_spot", dict(width=96, height=54)), ("c3_renault", dict(width=64, height=36)),
                 ("c4_spheres", dict(width=64, height=36, grid=20)), ("random_scene", dict(width=64, height=32, aperture=0.2)),
                 ("random_scene", dict(width=64, height=32, ground="checker"))]:
    desc = scenes.WORKLOADS[name](**kw)
    sky = (name == "random_scene")
    s = Scene(desc)
    for prec in (FAST_F32, EXACT_F64):
        integ = CudaPixelIntegrator(s, precision=prec, seed=1)
        a = integ.Sample(2)
        assert np.isfinite(a).all()
    integ = CudaPixelIntegrator(s, precision=FAST_F32, seed=1)
    for fl in (_lib.SAMPLE_REFERENCE_STREAM, _lib.SAMPLE_COUNT_OWN_TREE, _lib.SAMPLE_F32_PRIMARY) + (() if sky else (_lib.SAMPLE_COUNT_TRAVERSAL,)):
        integ.Sample(1, flags=fl)
    uv = np.random.default_rng(0).random((5000, 2))
    s.TracePrimary(uv, precision=FAST_F32); s.TracePrimary(uv, precision=EXACT_F64)
    org = np.random.default_rng(1).uniform(-1, 1, (4000, 3)) + [0, 1, 0]
    d = np.random.default_rng(2).normal(size=(4000, 3)); d[:2000, 1] = 0.0          # axis-parallel: the hybrid's exact fixup
    s.Hit(org, d / np.linalg.norm(d, axis=1)[:, None], 1e-5, 1e7, precision=FAST_F32)
    s.Hit(org, d / np.linalg.norm(d, axis=1)[:, None], 1e-5, 2.0, precision=FAST_F32, any_hit=True)
    film = Film(s)
    film.GetFrame(integ, 1); film.PostProcess(); film.close()
    for r in range(2):
        CudaPixelIntegrator(s, precision=FAST_F32, seed=1, tile_size=16, rank=r, world=2).SampleF32(1)
        CudaPixelIntegrator(s, precision=FAST_F32, seed=1, tile_size=16, rank=r, world=2).Sample(1, flags=_lib.SAMPLE_STRIPES)
    tex = [np.zeros((desc.width, desc.height, 4)) for _ in range(2)]
    for t in tex:
        _lib.check(_lib.load().mfx_host_register(_lib.ptr(t), t.nbytes))
    for k in range(3):
        integ.SampleAsync(1, tex[k % 2], first_sample=k)
    integ.Wait(); integ.Wait()
    for t in tex:
        _lib.load().mfx_host_unregister(_lib.ptr(t))
    m = MultiGpuPixelIntegrator(desc, precision=FAST_F32, seed=1)
    m.Sample(1); m.close()
    s.close()
    print("ok", name, flush=True)
