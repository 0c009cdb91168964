"""Headless driver: `python -m mafrixraytracing_b200.render scene.xml --frames 16 --spp 1 --out cornell`.

The window loop of RenderTest/Sample/RayTracing4.fs:73-80 without the window: InitSceneState (here: ingest.py),
`new Scene(state)`, then per displayed frame `film.GetFrame(pixelIntegrator, spp)` (Scene.fs:331-333) and, at the
end, the tone-mapped RGBA8 buffer (Scene.fs:315-330) as PNG plus the accumulated radiance as PFM.

`python -m mafrixraytracing_b200.render sphere-sample --width 400 --height 200 --frames 1 --spp 9 --out spheres` renders
the other sample, DoRayTrace of RenderTest/Sample/RayTracing.fs:417-473 (RandomScene, RayTraceCamera, GetColor, ns = 9),
whose pixel loop is commented out in the reference: the PNG is its sqrt / 255.99 / vertically flipped screen (:456-460)."""
import argparse
import os
import sys

import numpy as np

from . import Scene, CudaPixelIntegrator, Film, MultiGpuPixelIntegrator, MultiGpuFilm, EXACT_F64, FAST_F32
from .imageio import texture_to_rows, write_pfm, write_png
from .ingest import init_scene_state


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("scene", help="XML scene description (the reference's Scene.xml format), or `sphere-sample`")
    ap.add_argument("--width", type=int, default=400, help="sphere-sample only: nx (RayTracing.fs:423)")
    ap.add_argument("--height", type=int, default=200, help="sphere-sample only: ny (RayTracing.fs:424)")
    ap.add_argument("--frames", type=int, default=16)
    ap.add_argument("--spp", type=int, default=1, help="samples per pixel and frame (Scene.Render uses 1)")
    ap.add_argument("--exact", action="store_true", help="MFX_EXACT_F64 instead of MFX_FAST_F32")
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--out", default="frame")
    ap.add_argument("--gpus", type=int, default=None, help="the same loop over the first N devices (MultiGpuFilm)")
    a = ap.parse_args(argv)
    sky = (a.scene == "sphere-sample")
    if sky:
        from .scenes import random_scene
        desc = random_scene(width=a.width, height=a.height, seed=a.seed + 41)
    else:
        with open(a.scene, "r", encoding="utf-8-sig") as fh:
            desc = init_scene_state(fh.read(), base_dir=os.path.dirname(os.path.abspath(a.scene)))
    precision = EXACT_F64 if a.exact else FAST_F32
    if a.gpus:                          # one host thread, N devices: each keeps the Film of its own stripes
        scene = integ = MultiGpuPixelIntegrator(desc, n_devices=a.gpus, precision=precision, seed=a.seed)
        if integ.n_devices < a.gpus:
            integ.close()
            raise SystemExit(f"--gpus {a.gpus} but {integ.n_devices} device(s) visible")
        film = MultiGpuFilm(integ)
        get_frame = lambda f: film.GetFrame(a.spp, first_sample=f * a.spp, download=(f + 1 == a.frames))
    else:
        scene = Scene(desc)
        integ = CudaPixelIntegrator(scene, precision=precision, seed=a.seed)
        film = Film(scene)
        get_frame = lambda f: film.GetFrame(integ, a.spp, first_sample=f * a.spp)
    rays = ms = 0.0
    for f in range(a.frames):
        target = get_frame(f)
        rays += integ.stats["closest_rays"] + integ.stats["shadow_rays"]
        ms += integ.stats["ms_total"]
    rows = texture_to_rows(target)[:, :, :3].astype(np.float32)
    if sky:
        rows = rows[::-1]               # row j of this texture grows upwards (v runs along `vertical`): top row first
    write_pfm(a.out + ".pfm", rows)
    write_png(a.out + ".png", film.PostProcess())
    film.close()
    print(f"{desc.width}x{desc.height}, {len(desc.prims)} shapes, {a.frames} frames x {a.spp} spp: "
          f"{rays / 1e6:.1f} Mrays in {ms:.1f} ms ({rays / max(ms, 1e-9) / 1e3:.0f} Mrays/s) -> {a.out}.pfm, {a.out}.png")
    scene.close()
    return 0


if __name__ == "__main__":
    sys.exit(main())
