"""MultiGpuFilm (mfx_multi_film_*): the progressive Film over several GPUs, each device accumulating, dividing and
tone-mapping its own column stripes.  Every result must equal the one-GPU Film's bit for bit: the per-pixel arithmetic is
the same and the RNG is keyed on the absolute pixel and sample.  Every case runs on device 0 alone and on every visible
device."""
import os
import subprocess
from ctypes import byref, c_double

import numpy as np
import pytest

from mafrixraytracing_b200 import (scenes, Scene, CudaPixelIntegrator, Film, MultiGpuPixelIntegrator, MultiGpuFilm,
                                   MafrixError, EXACT_F64, FAST_F32)
from mafrixraytracing_b200 import _lib

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _device_sets():
    n = _lib.load().mfx_device_count()
    return ([0], list(range(n))) if n > 1 else ([0],)


def _count(film):
    fc = c_double()
    _lib.check(_lib.load().mfx_film_frame_count(film._h, byref(fc)))
    return fc.value


def _single_run(desc, precision, seed, frames, spp):
    """The one-GPU Film: every frame's target, its count, the screen, and a fresh film for the caller."""
    s = Scene(desc)
    integ = CudaPixelIntegrator(s, precision=precision, seed=seed)
    film = Film(s)
    targets, counts = [], []
    for _ in range(frames):
        targets.append(film.GetFrame(integ, spp).copy())
        counts.append(_count(film))
    return targets, counts, film.PostProcess(), (s, integ, film)


SCENES = [("cornell", dict(width=24, height=40)),            # 24 columns: devices beyond the second own no stripe
          ("c1_cube", dict(width=333, height=120)),          # partial last stripe
          ("c2_spot", dict(width=480, height=270)),          # mode A
          ("c3_renault", dict(width=480, height=270)),       # mode B
          ("random_scene", dict(width=200, height=100))]     # the sphere sample: display transform with its vertical flip


@pytest.mark.parametrize("name,kw", SCENES, ids=[n for n, _ in SCENES])
def test_multi_film_frames_and_screen_equal_the_single_gpu_film(name, kw):
    desc = scenes.WORKLOADS[name](**kw)
    want, counts, screen, (s, integ, film) = _single_run(desc, FAST_F32, 3, 4, 2)
    film.GetFrame(integ, 2)
    screen5 = film.PostProcess()
    for devs in _device_sets():
        m = MultiGpuPixelIntegrator(desc, devices=devs, precision=FAST_F32, seed=3)
        mf = MultiGpuFilm(m)
        for k in range(4):
            got = mf.GetFrame(2)
            assert np.array_equal(got, want[k]), f"{name} on {devs}: frame {k} differs"
            assert mf.FrameCount() == counts[k]
        assert np.array_equal(mf.PostProcess(), screen)
        assert mf.GetFrame(2, download=False) is None                # texture = NULL: the target stays on the devices
        assert np.array_equal(mf.PostProcess(), screen5)
        m.close()
    s.close()


def test_multi_film_exact_precision_equals_the_single_gpu_film():
    desc = scenes.cornell(width=64, height=48)
    want, counts, screen, (s, _, _) = _single_run(desc, EXACT_F64, 8, 3, 1)
    for devs in _device_sets():
        m = MultiGpuPixelIntegrator(desc, devices=devs, precision=EXACT_F64, seed=8)
        mf = MultiGpuFilm(m)
        for k in range(3):
            assert np.array_equal(mf.GetFrame(1), want[k]) and mf.FrameCount() == counts[k]
        assert np.array_equal(mf.PostProcess(), screen)
        m.close()
    s.close()


def test_multi_film_checkpoint_resumes_across_device_counts():
    desc = scenes.c1_cube(width=333, height=120)
    want, _, screen, (s, integ, film) = _single_run(desc, FAST_F32, 5, 5, 2)
    film.Reset()
    for _ in range(3):
        film.GetFrame(integ, 2)
    single_sum, single_count = film.Export()
    assert single_count == 3.0
    sets = _device_sets()
    for src in sets:
        m = MultiGpuPixelIntegrator(desc, devices=src, precision=FAST_F32, seed=5)
        mf = MultiGpuFilm(m)
        for _ in range(3):
            mf.GetFrame(2)
        saved, count = mf.Export()
        assert count == 3.0 and np.array_equal(saved, single_sum)
        # multi -> one-GPU Film
        s2 = Scene(desc)
        f2 = Film(s2)
        f2.Import(saved, count)
        i2 = CudaPixelIntegrator(s2, precision=FAST_F32, seed=5)
        for _ in range(2):
            resumed = f2.GetFrame(i2, 2).copy()
        assert np.array_equal(resumed, want[4]) and np.array_equal(f2.PostProcess(), screen)
        s2.close()
        for dst in sets:
            # multi -> multi (the same device count and the other one), and one-GPU Film -> multi
            for sum_in, count_in in ((saved, count), (single_sum, single_count)):
                d = MultiGpuPixelIntegrator(desc, devices=dst, precision=FAST_F32, seed=5)
                df = MultiGpuFilm(d)
                df.Import(sum_in, count_in)
                assert df.FrameCount() == 3.0
                for _ in range(2):
                    resumed = df.GetFrame(2).copy()
                assert np.array_equal(resumed, want[4]) and np.array_equal(df.PostProcess(), screen)
                d.close()
        with pytest.raises(ValueError):
            mf.Import(saved[:, :-1], count)
        m.close()
    s.close()


def test_multi_film_reset_starts_over():
    desc = scenes.c2_spot(width=480, height=270)
    want, _, _, (s, _, _) = _single_run(desc, FAST_F32, 2, 1, 1)
    for devs in _device_sets():
        m = MultiGpuPixelIntegrator(desc, devices=devs, precision=FAST_F32, seed=2)
        mf = MultiGpuFilm(m)
        mf.GetFrame(1)
        mf.GetFrame(1)
        mf.Reset()
        assert mf.FrameCount() == 0.0
        assert np.array_equal(mf.GetFrame(1), want[0]) and mf.FrameCount() == 1.0
        m.close()
    s.close()


def test_multi_film_lifetime_and_concurrency_rules():
    desc = scenes.cornell(width=96, height=64)
    want, _, _, (s, _, _) = _single_run(desc, FAST_F32, 4, 2, 2)
    lib = _lib.load()
    for devs in _device_sets():
        m = MultiGpuPixelIntegrator(desc, devices=devs, precision=FAST_F32, seed=4)
        mf = MultiGpuFilm(m)
        assert np.array_equal(mf.GetFrame(2), want[0])
        m.Sample(3, first_sample=40)                                  # a plain Sample between film frames
        assert np.array_equal(mf.GetFrame(2), want[1]) and mf.FrameCount() == 2.0
        tex = np.zeros((desc.width, desc.height, 4))
        _lib.check(lib.mfx_host_register(_lib.ptr(tex), tex.nbytes))
        try:
            m.SampleAsync(2, tex)
            with pytest.raises(MafrixError):
                mf.GetFrame(2)                                        # one job in flight per handle
            with pytest.raises(MafrixError):
                mf.PostProcess()
            m.Wait()
        finally:
            lib.mfx_host_unregister(_lib.ptr(tex))
        assert mf.FrameCount() == 2.0
        saved, _ = mf.Export()
        assert np.array_equal(saved[:, :, :3] / 2.0, want[1][:, :, :3])
        with pytest.raises(MafrixError):
            _lib.check(lib.mfx_multi_destroy(m._h))                   # a film of the handle is alive
        mf.close()
        assert lib.mfx_multi_destroy(m._h) == 0
        m._h = None
    # MultiGpuPixelIntegrator.close() takes its films down first
    m = MultiGpuPixelIntegrator(desc, devices=[0], precision=FAST_F32, seed=4)
    mf = MultiGpuFilm(m)
    m.close()
    assert m._h is None and mf._h is None
    s.close()


def test_cpp_and_python_hosts_render_through_the_multi_film(tmp_path):
    """host/render_test --gpus N and `python -m mafrixraytracing_b200.render --gpus N` give the one-GPU run's PFM and
    screen.  With one device the C++ host refuses --gpus 2."""
    exe = os.path.join(ROOT, "host", "render_test")
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "host"), "-s"])
    n = _lib.load().mfx_device_count()
    if n < 2:
        r = subprocess.run([exe, "--gpus", "2", "--frames", "1", "--size", "64x48", "--out", str(tmp_path / "x")],
                           capture_output=True, text=True)
        assert r.returncode == 1 and "device(s) visible" in r.stderr
    a = str(tmp_path / "one")
    subprocess.check_call([exe, "--frames", "3", "--spp", "2", "--size", "250x90", "--out", a])
    for g in sorted({1, n}):
        b = str(tmp_path / f"many{g}")
        subprocess.check_call([exe, "--frames", "3", "--spp", "2", "--size", "250x90", "--gpus", str(g), "--out", b])
        assert open(a + ".pfm", "rb").read() == open(b + ".pfm", "rb").read()
        assert open(a + ".ppm", "rb").read() == open(b + ".ppm", "rb").read()
    from mafrixraytracing_b200 import render
    args = ["sphere-sample", "--width", "120", "--height", "60", "--frames", "2", "--spp", "2"]
    assert render.main(args + ["--out", a]) == 0
    for g in sorted({1, n}):
        b = str(tmp_path / f"py{g}")
        assert render.main(args + ["--gpus", str(g), "--out", b]) == 0
        for ext in (".pfm", ".png"):
            assert open(a + ext, "rb").read() == open(b + ext, "rb").read()
