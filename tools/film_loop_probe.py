"""The reference's display loop (Scene.Render -> Film.GetFrame(integrator, 1) -> PostProcessAndToScreenBuffer) on N GPUs,
two ways, in one process, alternating:

  (a) host film: mfx_multi_sample into a pinned Color[w,h], then sum += frame, target = sum / frameCount and the ACES
      tone map in numpy on the host -- what a host without a multi-GPU Film has to do;
  (b) device film: mfx_multi_film_get_frame(texture = NULL) + mfx_multi_film_post_process -- only the RGBA8 screen
      crosses PCIe.

Reports ms per displayed frame for each arm (host clock around calls that end in a device synchronise), for N = 1 and
every larger device count visible, with the GPU name and power limit read in the same run.  Both arms render the same
samples, so their screens must be byte-equal: the run checks that too.

  python tools/film_loop_probe.py [--scene c2_spot] [--frames 50] [--warmup 5] [--rounds 3] [--out result.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from mafrixraytracing_b200 import scenes, MultiGpuPixelIntegrator, MultiGpuFilm, FAST_F32, _lib  # noqa: E402


def aces_rgba8(target_wh):
    """Scene.fs:273-289,315-330 on the host: ACES, sqrt, int(255.99 c) -> (height, width, 4) uint8."""
    v = np.transpose(target_wh[:, :, :3], (1, 0, 2))
    num = v * (2.51 * v + 0.03)
    den = v * (2.43 * v + 0.59) + 0.14
    out = np.empty(v.shape[:2] + (4,), np.uint8)
    out[:, :, :3] = (255.99 * np.sqrt(np.clip(num / den, 0.0, 1.0))).astype(np.int32).astype(np.uint8)
    out[:, :, 3] = 255
    return out


def gpu_info():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60)
        return [line.strip() for line in r.stdout.splitlines() if line.strip()]
    except (OSError, subprocess.SubprocessError) as e:
        return [f"nvidia-smi unavailable: {e}"]


def run(desc, n, frames, warmup, rounds):
    lib = _lib.load()
    m = MultiGpuPixelIntegrator(desc, n_devices=n, precision=FAST_F32, seed=1)
    m.Prepare()
    W, H = desc.width, desc.height
    frame = np.zeros((W, H, 4))
    screen = np.zeros((H, W, 4), np.uint8)
    _lib.check(lib.mfx_host_register(_lib.ptr(frame), frame.nbytes))
    _lib.check(lib.mfx_host_register(_lib.ptr(screen), screen.nbytes))
    film = MultiGpuFilm(m)
    host = {"sum": np.zeros((W, H, 4)), "count": 0}

    def host_frame():                      # arm (a)
        k = host["count"]
        m.Sample(1, first_sample=k, out=frame)
        host["count"] = k + 1
        host["sum"][:, :, :3] += frame[:, :, :3]
        target = host["sum"] / float(k + 1)
        return aces_rgba8(target)

    def device_frame():                    # arm (b)
        film.GetFrame(1, download=False)
        return film.PostProcess(out=screen)

    arms = {"a_host_film": host_frame, "b_device_film": device_frame}
    per = {k: [] for k in arms}
    try:
        for fn in arms.values():
            for _ in range(warmup):
                fn()
        for _ in range(rounds):
            for name, fn in arms.items():
                t = []
                for _ in range(frames):
                    t0 = time.perf_counter()
                    fn()
                    t.append((time.perf_counter() - t0) * 1e3)
                per[name].extend(t)
        # both arms have rendered the same samples: the screens must agree byte for byte
        host["sum"][:, :, 3] = 0.0
        equal = bool(np.array_equal(aces_rgba8(host["sum"] / float(host["count"])), film.PostProcess()))
        assert host["count"] == film.FrameCount()
    finally:
        film.close()
        lib.mfx_host_unregister(_lib.ptr(frame))
        lib.mfx_host_unregister(_lib.ptr(screen))
        m.close()
    res = {"n_devices": n, "frames_timed": frames * rounds, "screens_equal": equal}
    for name, t in per.items():
        a = np.asarray(t)
        res[name] = {"median_ms": round(float(np.median(a)), 3), "mean_ms": round(float(a.mean()), 3),
                     "p90_ms": round(float(np.percentile(a, 90)), 3)}
    return res


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--scene", default="c2_spot")
    ap.add_argument("--width", type=int, default=1920)
    ap.add_argument("--height", type=int, default=1080)
    ap.add_argument("--frames", type=int, default=50, help="timed frames per arm and round")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3, help="alternations of the two arms")
    ap.add_argument("--max-devices", type=int, default=0)
    ap.add_argument("--out", default=None, help="also write the JSON result here")
    a = ap.parse_args(argv)
    n_vis = _lib.load().mfx_device_count()
    if n_vis <= 0:
        raise SystemExit("no CUDA device visible: this probe measures on the GPU only")
    top = min(n_vis, a.max_devices) if a.max_devices > 0 else n_vis
    desc = scenes.WORKLOADS[a.scene](width=a.width, height=a.height)
    result = {"scene": a.scene, "size": f"{a.width}x{a.height}", "spp_per_frame": 1, "gpus": gpu_info(), "runs": []}
    for n in range(1, top + 1):
        r = run(desc, n, a.frames, a.warmup, a.rounds)
        print(json.dumps(r), flush=True)
        result["runs"].append(r)
    line = json.dumps(result)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(line + "\n")
    return 0 if all(r["screens_equal"] for r in result["runs"]) else 1


if __name__ == "__main__":
    sys.exit(main())
