#!/usr/bin/env python3
"""bench.py -- the headline measurement: Mrays/s (primary + secondary) of the path-tracing hot
path on BASELINE.json configs[1]: spot (cow OBJ) 1920x1080, 64 spp, max depth 5, diffuse + area
light (SURVEY.md 8(d) "C2"), one step = one IPixelIntegrator.Sample(64) of the whole frame.

  python bench.py --gpus 1 --steps K --warmup W          this repo's CUDA path (libmafrix_cuda)
  torchrun ... bench.py --gpus N ...                     frame stripe-sharded over N GPUs (one process each) + NCCL gather
  python bench.py --impl reference ...                   the reference's CPU algorithm (the oracle
                                                         restatement; .NET is not in this image)
  --dump-outputs DIR                                     also write the frame of the last timed step (DIR/color.npy)

value   : whole-job Mrays/s, scene + path state resident in HBM, result left in HBM (device timed)
e2e     : same metric through the reference-facing call with HOST buffers -- scene upload + Sample -> Color[w,h] on the
          host, copies inside the timed region.  N = 1: mfx_scene_create + mfx_pixel_integrator_sample; N > 1: what a
          single-threaded host (the reference's shape) calls: mfx_multi_create + mfx_multi_sample over the N GPUs, from
          rank 0 alone while the other ranks wait on a CPU barrier
roofline: closest-hit traversal kernel.  The scene of this workload is cache resident, so the bound is the rate at which
          the L1 turns divergent 32-byte sectors around: achieved = bytes of records + primitives the kernel requests per
          ray (instrumented run on its own tree) x rays / CUDA-event time, peak = the same access pattern measured live on
          this GPU by tools/peaks_cache.  `hbm_definition` keeps SURVEY 8(d)'s figure (reference-tree records against the
          HBM copy bandwidth) -- labelled: it exceeds 1 because those bytes never leave the caches; `dram` is the DRAM
          traffic ncu measured for the whole step against the 64 B/ray queue budget and the HBM peak
configs : BASELINE configs[2..4] at their stated size through the same device-timed path
primary : the id-exact bounce-0 kernel (hybrid: f32 boxes, f64 primitive tests) against f32 primitive tests, primary rays alone
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "Mrays/s (primary+secondary)"
WORKLOAD = "c2_spot: spot 5856 tris + floor + back wall, 1920x1080, 64 spp, max depth 5, PathIntegrator, 1 quad light"
SPP = 64
REF_SPP = 2            # bounded sample for the CPU arms: same frame, 2 spp per step


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="mafrix", choices=["mafrix", "reference"])
    ap.add_argument("--spp", type=int, default=SPP)
    ap.add_argument("--workload", default="c2_spot")
    ap.add_argument("--precision", default="fast", choices=["fast", "exact"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the C3/C4/C5 table (about a minute at N=1)")
    ap.add_argument("--no-primary", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the Color[w,h] frame of the last timed step to DIR/color.npy (float32) to compare builds")
    return ap.parse_args()


DUMP_LIMIT = 64 << 20


def dump_outputs(out_dir, color):
    """Writes Color[w,h] as float32.  A frame above DUMP_LIMIT (the 4K configs) keeps every s-th pixel along both axes,
    with the smallest s that fits, so the same arguments always select the same pixels."""
    a = color.astype(np.float32)
    s = 1
    while a[::s, ::s].nbytes > DUMP_LIMIT:
        s += 1
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "color.npy"), np.ascontiguousarray(a[::s, ::s]))
    print(f"bench: wrote {out_dir}/color.npy, Color[w,h] of the last timed step, pixel stride {s}", file=sys.stderr, flush=True)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md, file absent)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [x.strip() for x in line.split(",")]))

    def count_since(self, t0):
        return sum(1 for t, _ in list(self.rows) if t >= t0)

    def stop(self, t0=0.0):
        """Statistics of the samples taken at or after t0 (the start of the timed region)."""
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for t, r in self.rows:
            if t < t0:
                continue
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def b_ray(nodes, tris, spheres, rays):
    return (32.0 * nodes + 48.0 * tris + 16.0 * spheres) / max(rays, 1) + 64.0


def run_reference(args, rank, world):
    """The reference's own CPU implementation of the path, restated (oracle/mafrix_oracle.c, f64,
    exhaustive both-children traversal, recursion to depth -1), OpenMP over pixels on all host
    cores like Array.Parallel.iter (Integrators.fs:164).  A step = the same frame at REF_SPP spp."""
    if rank != 0:
        return
    from mafrixraytracing_b200 import scenes
    from oracle import oracle
    desc = scenes.WORKLOADS[args.workload]()
    o = oracle.OracleScene(desc)
    cores = host_cores()              # torchrun exports OMP_NUM_THREADS=1: ask for every core explicitly
    tex = np.zeros((desc.width, desc.height, 4))
    for _ in range(args.warmup):
        o.sample(REF_SPP, seed=1, out=tex, threads=cores)
    t0 = time.perf_counter()
    for k in range(args.steps):
        o.sample(REF_SPP, seed=1, first_sample=k * REF_SPP, out=tex, threads=cores)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, tex)
    # rays per step: count them with one instrumented (slower, untimed) step
    _, st = o.sample(REF_SPP, seed=1, stats=True, threads=cores)
    rays = st["closest_rays"] + st["wasted_rays"] + st["shadow_rays"]
    val = rays * args.steps / dt / 1e6
    sample = f"full 1920x1080 frame at {REF_SPP} spp per step (config is 64 spp; cost is linear in spp), {rays} rays/step incl. the reference's wasted depth -1 query"
    line = {"metric": METRIC, "value": val, "unit": "Mrays/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "impl": "reference",
            "config": {"workload": WORKLOAD, "sample": sample},
            "cpu_baseline": {"value": val, "unit": "Mrays/s", "cores": cores, "kind": "port", "sample": sample,
                             "spp_per_s": REF_SPP * args.steps / dt},
            "e2e": {"value": val, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
            "note": "C restatement of the reference CPU path (the F# original needs .NET, absent here); a reported baseline, not the target"}
    print(json.dumps(line), flush=True)


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def cpu_baseline(desc):
    from oracle import oracle
    o = oracle.OracleScene(desc)
    cores = host_cores()
    _, st = o.sample(1, seed=1, stats=True, threads=cores)      # instrumented: rays per spp
    rays_per_spp = st["closest_rays"] + st["wasted_rays"] + st["shadow_rays"]
    n = 4
    t0 = time.perf_counter()
    o.sample(n, seed=1, first_sample=1, threads=cores)
    dt = time.perf_counter() - t0
    return {"value": rays_per_spp * n / dt / 1e6, "unit": "Mrays/s", "cores": cores, "kind": "port",
            "sample": f"full 1920x1080 frame at {n} spp ({rays_per_spp * n} rays incl. the wasted depth -1 queries), {dt:.1f} s on {cores} threads",
            "spp_per_s": n / dt, "ref_nodes_per_ray": st["ref_nodes"] / rays_per_spp, "ref_prims_per_ray": st["ref_prims"] / rays_per_spp}


def cache_peaks():
    """On-chip bandwidth of THIS GPU for the traversal kernel's access pattern (divergent 256-bit record loads), measured
    live by tools/peaks_cache (built by __graft_entry__.build())."""
    exe = os.path.join(ROOT, "tools", "peaks_cache")
    if not os.path.exists(exe):
        return None
    try:
        out = subprocess.run([exe], capture_output=True, text=True, timeout=120)
        return json.loads(out.stdout.strip().splitlines()[-1]) if out.returncode == 0 else None
    except Exception:
        return None


def load_traffic():
    """DRAM bytes per launch / per step of the bench configuration, from the committed ncu capture (profiles/)."""
    for name in ("r02_traffic.json", "roofline_traffic.json"):
        p = os.path.join(ROOT, "profiles", name)
        if os.path.exists(p):
            d = json.load(open(p))
            d["file"] = "profiles/" + name
            return d
    return {}


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    dbg = (lambda *a: print(f"[bench rank {rank}]", *a, file=sys.stderr, flush=True)) if os.environ.get("BENCH_DEBUG") else (lambda *a: None)
    dbg("start", sys.argv)
    import torch
    import torch.distributed as dist
    from mafrixraytracing_b200 import scenes, Scene, CudaPixelIntegrator, MultiGpuPixelIntegrator, Bvh, EXACT_F64, FAST_F32, _lib
    from mafrixraytracing_b200 import dist as mdist

    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")     # a box that sets NCCL_DEBUG=VERSION must not write into the JSON stream
    torch.cuda.set_device(local_rank)
    cpu_group = None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group(backend="nccl", device_id=torch.device("cuda", local_rank))
        cpu_group = dist.new_group(backend="gloo")       # waits that must not occupy a GPU (rank 0 drives all of them in the e2e leg)
    dbg("process group up")
    prec = FAST_F32 if args.precision == "fast" else EXACT_F64
    desc = scenes.WORKLOADS[args.workload]()
    bvh = Bvh.Build(desc.prims)                                 # host, one-off (kept on the host by the north star)
    scene = Scene(desc, bvh=bvh, device=local_rank)
    sharded = mdist.ShardedPixelIntegrator(scene, rank, world, precision=prec, seed=1, stripe=mdist.STRIPE)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")           # > 126 MB L2

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def cpu_barrier():
        if world > 1:
            dist.barrier(group=cpu_group)

    def timed_step(integ, spp, k=0):
        flush.fill_(k & 0xff)                                   # L2 flush between iterations
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        integ.Sample(spp, first_sample=0)                       # render this rank's stripes + NCCL gather of the owned stripes to rank 0
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1), dict(integ.stats)

    def step(k):
        return timed_step(sharded, args.spp, k)

    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()          # nvidia-smi needs ~0.2 s to deliver its first row: start it ahead, keep rows from wall0 on
    for k in range(max(args.warmup, 3)):
        step(k)
    sync_all()
    wall0 = time.perf_counter()
    ms_steps, stats = [], []
    for k in range(args.steps):
        ms, st = step(k)
        ms_steps.append(ms)
        stats.append(st)
    sync_all()
    wall = time.perf_counter() - wall0
    # the later legs render into the same frame
    last_frame = sharded.frame.cpu().numpy() if args.dump_outputs and rank == 0 else None
    # a timed region shorter than a few sampling periods (8 GPUs: 5 x 10 ms) may hold no sample: keep the same load
    # running, untimed, until three rows exist (all ranks take part: the step has a collective)
    extra = 0
    while world >= 1:
        need = torch.tensor([1 if (rank == 0 and clocks.proc and clocks.count_since(wall0) < 3 and extra < 400) else 0], device="cuda")
        if world > 1:
            dist.broadcast(need, 0)
        if not int(need.item()):
            break
        step(0)
        extra += 1
    clk = clocks.stop(wall0) if rank == 0 else None
    if last_frame is not None:
        dump_outputs(args.dump_outputs, last_frame)
    if clk is not None:
        clk["window"] = "timed region" if extra == 0 else f"timed region + {extra} identical untimed steps (region shorter than the sampling period)"

    def aggregate(rays_rank, t_rank):
        if world > 1:
            tt = torch.tensor([t_rank], dtype=torch.float64, device="cuda")
            rr = torch.tensor([float(rays_rank)], dtype=torch.float64, device="cuda")
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            dist.all_reduce(rr, op=dist.ReduceOp.SUM)
            return rr.item(), tt.item()
        return float(rays_rank), t_rank

    dbg("timed region done")
    rays_all, t_all = aggregate(sum(s["closest_rays"] + s["shadow_rays"] for s in stats), sum(ms_steps))
    value = rays_all / t_all / 1e3                               # rays / ms / 1e3 = Mrays/s

    # ---- end to end through the reference-facing call, host buffers
    e2e = None
    if not args.no_e2e:
        h2d = desc.prims.nbytes + desc.materials.nbytes + bvh.nodes.nbytes + bvh.indices.nbytes + 12 * 8 + 18 * 8
        rays_e2e, t_e2e, d2h = 0.0, 0.0, 0
        texs = []
        if rank == 0:
            # the host keeps its Texture2D<Color> for its lifetime (Integrators.fs:147): pinned once so the per-frame
            # download is a direct DMA (INTEGRATION.md, mfx_host_register).  Two of them: frame k downloads while frame k+1
            # renders (mfx_pixel_integrator_sample_async), the pipelined form of the reference's frame-after-frame loop
            for _ in range(2):
                t = np.zeros((desc.width, desc.height, 4), dtype=np.float64)
                _lib.check(_lib.load().mfx_host_register(_lib.ptr(t), t.nbytes))
                texs.append(t)
            d2h = texs[0].nbytes
        cpu_barrier()                                            # N > 1: ranks 1.. hold no GPU work while rank 0 drives every device
        if rank == 0 and world == 1:
            def pipelined(n_steps):
                """n_steps frames, each through its own `new Scene(state)`: H2D of the flattened scene, Sample, D2H of Color[w,h]."""
                rays, prev = 0.0, None
                for k in range(n_steps):
                    sc = Scene(desc, bvh=bvh, device=local_rank)     # H2D: prims, tree, materials -> flattened layouts
                    integ = CudaPixelIntegrator(sc, precision=prec, seed=1)
                    integ.SampleAsync(args.spp, texs[k % 2])         # kernels + D2H enqueued; returns at once
                    if prev is not None:
                        prev[1].Wait()                               # frame k-1 complete on the host
                        rays += prev[1].stats["closest_rays"] + prev[1].stats["shadow_rays"]
                        prev[0].close()
                    prev = (sc, integ)
                prev[1].Wait()
                rays += prev[1].stats["closest_rays"] + prev[1].stats["shadow_rays"]
                prev[0].close()
                return rays
            pipelined(2)                                             # untimed: allocates the path state of two frames in flight
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            rays_e2e = pipelined(args.steps)
            t_e2e = time.perf_counter() - t0
            # the same step without pipelining (one blocking call per frame), for reference
            t0 = time.perf_counter()
            for k in range(args.steps):
                sc = Scene(desc, bvh=bvh, device=local_rank)
                CudaPixelIntegrator(sc, precision=prec, seed=1).Sample(args.spp, out=texs[0])
                sc.close()
            t_block = time.perf_counter() - t0
        elif rank == 0:
            def one_blocking():
                m = MultiGpuPixelIntegrator(desc, devices=list(range(world)), bvh=bvh, precision=prec, seed=1)
                m.Sample(args.spp, out=texs[0])                  # every device DMAs its stripes into the one host texture
                st = m.stats
                m.close()
                return st["closest_rays"] + st["shadow_rays"]

            def pipelined_multi(n_steps):
                """n_steps frames, each through its own mfx_multi_create: frame k renders and downloads while the host thread
                creates the replicas of frame k+1 and posts it (mfx_multi_sample_async / mfx_multi_wait); on every device the
                kernels of frame k+1 are ordered behind those of frame k by an event, everything else overlaps."""
                rays, prev, stamps = 0.0, None, [time.perf_counter()]
                for k in range(n_steps):
                    m = MultiGpuPixelIntegrator(desc, devices=list(range(world)), bvh=bvh, precision=prec, seed=1)
                    m.SampleAsync(args.spp, texs[k % 2])
                    if prev is not None:
                        prev.Wait()
                        stamps.append(time.perf_counter())
                        rays += prev.stats["closest_rays"] + prev.stats["shadow_rays"]
                        prev.close()
                    prev = m
                prev.Wait()
                stamps.append(time.perf_counter())
                rays += prev.stats["closest_rays"] + prev.stats["shadow_rays"]
                prev.close()
                dbg("pipelined_multi frame completion intervals, ms: " + " ".join(f"{1e3 * (b - a):.1f}" for a, b in zip(stamps[:-1], stamps[1:])))
                return rays
            one_blocking(); pipelined_multi(3)                       # untimed: contexts, path state of two frames in flight
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            rays_e2e = pipelined_multi(args.steps)
            t_e2e = time.perf_counter() - t0
            t0 = time.perf_counter()
            for k in range(args.steps):
                one_blocking()
            t_block = time.perf_counter() - t0
        if rank == 0:
            for t in texs:
                _lib.load().mfx_host_unregister(_lib.ptr(t))
        cpu_barrier()
        if rank == 0:
            e2e = {"value": rays_e2e / t_e2e / 1e6, "unit": "Mrays/s", "h2d_bytes_per_step": int(h2d * world), "d2h_bytes_per_step": int(d2h),
                   "ms_per_step": t_e2e / args.steps * 1e3,
                   "blocking_ms_per_step": t_block / args.steps * 1e3 if t_block else None,
                   "call": "per frame: mfx_scene_create + mfx_pixel_integrator_sample_async -> pinned Color[w,h] f64, mfx_pixel_integrator_wait on the "
                           "previous frame (two frames in flight: download k beside render k+1); blocking_ms_per_step = the same with "
                           "mfx_pixel_integrator_sample" if world == 1 else
                           f"per frame: mfx_multi_create + mfx_multi_sample_async from ONE host thread over {world} GPUs (scene replicated per device, "
                           "every device DMAs its column stripes into the pinned host texture), mfx_multi_wait on the previous frame; "
                           "blocking_ms_per_step = the same with mfx_multi_sample; ranks 1.. idle on a CPU barrier"}

    dbg("e2e done")
    # ---- roofline of the dominant kernel (closest-hit traversal), rank 0's share
    roof, cpu, primary = None, None, None
    if rank == 0:
        integ = sharded.integ
        fl = sharded.flags
        integ.SampleDeviceColor(2, sharded.frame.data_ptr(), flags=fl | _lib.SAMPLE_COUNT_TRAVERSAL)     # instrumented, untimed
        cs = integ.stats
        bc = b_ray(cs["nodes"][0], cs["tris"][0], cs["spheres"][0], cs["closest_rays"])
        bs = b_ray(cs["nodes"][1], cs["tris"][1], cs["spheres"][1], cs["shadow_rays"])
        ext_ms = sum(s["ms_extend"] for s in stats)
        ext_rays = sum(s["closest_rays"] for s in stats)
        ext_launches = sum(s["launches_extend"] for s in stats)
        sh_ms = sum(s["ms_shadow"] for s in stats)
        sh_rays = sum(s["shadow_rays"] for s in stats)
        step_ms = sum(s["ms_total"] for s in stats)
        hbm_peak, how = peaks()
        traffic = load_traffic()
        dev_bytes = scene.device_bytes()
        hbm_def = {"bytes_per_ray_closest": bc, "bytes_per_ray_shadow": bs,
                   "nodes_per_ray": [cs["nodes"][0] / max(cs["closest_rays"], 1), cs["nodes"][1] / max(cs["shadow_rays"], 1)],
                   "tris_per_ray": [cs["tris"][0] / max(cs["closest_rays"], 1), cs["tris"][1] / max(cs["shadow_rays"], 1)],
                   "achieved": ext_rays * bc / (ext_ms * 1e-3) / 1e9, "peak": hbm_peak, "peak_source": how,
                   "frac": ext_rays * bc / (ext_ms * 1e-3) / 1e9 / hbm_peak,
                   "whole_step_achieved_gbs": (ext_rays * bc + sh_rays * bs) / (step_ms * 1e-3) / 1e9,
                   "note": "SURVEY 8(d) / north star definition: 32 B/node + 48 B/tri + 16 B/sphere + 64 B of records an ordered, t-shrinking "
                           "traversal of the REFERENCE's median-split tree touches, against the HBM copy bandwidth.  NOT a roofline of the "
                           "shipped kernel: it walks its own SAH tree (a quarter of those records) and the scene never leaves the caches, "
                           "so the figure exceeds 1; kept for comparability with round 1"}
        roof = {"kernel": "k_f_trace6<closest> (BVH traversal of the extend queue)" if prec == FAST_F32 else "k_x_extend",
                "avg_launch_ms": ext_ms / max(ext_launches, 1), "launches": ext_launches, "share_of_step": ext_ms / max(step_ms, 1e-9),
                "extend_mrays_s": ext_rays / ext_ms / 1e3, "shadow_mrays_s": sh_rays / max(sh_ms, 1e-9) / 1e3,
                "scene_fast_bytes": dev_bytes["fast"], "hbm_definition": hbm_def}
        if prec == FAST_F32:
            # what the shipped kernel really requests: 128 B four-child records + 48 B triangle slots of its own tree
            integ.SampleDeviceColor(2, sharded.frame.data_ptr(), flags=fl | _lib.SAMPLE_COUNT_OWN_TREE)
            os_ = integ.stats
            rec = [os_["nodes"][0] / max(os_["closest_rays"], 1), os_["nodes"][1] / max(os_["shadow_rays"], 1)]
            tri = [os_["tris"][0] / max(os_["closest_rays"], 1), os_["tris"][1] / max(os_["shadow_rays"], 1)]
            sph = [os_["spheres"][0] / max(os_["closest_rays"], 1), os_["spheres"][1] / max(os_["shadow_rays"], 1)]
            own_bc = 128.0 * rec[0] + 48.0 * tri[0] + 16.0 * sph[0]
            own_bs = 128.0 * rec[1] + 48.0 * tri[1] + 16.0 * sph[1]
            ach = ext_rays * own_bc / (ext_ms * 1e-3) / 1e9
            cp = cache_peaks()          # rank 0's GPU; the other ranks wait at the next barrier
            roof.update({"records_per_ray": rec, "tris_per_ray": tri, "spheres_per_ray": sph,
                         "bytes_per_ray_closest": own_bc, "bytes_per_ray_shadow": own_bs,
                         "algorithmic_bytes_per_launch": ext_rays * own_bc / max(ext_launches, 1),
                         "achieved": ach, "unit": "GB/s",
                         "shadow_achieved": sh_rays * own_bs / max(sh_ms * 1e-3, 1e-12) / 1e9})
            if cp:
                # the scene (records + slots) is far below L2 size; the part of it a block keeps in its L1 is served at the
                # 64 KB figure, the rest at the L2 figure: the L1-resident figure is the ceiling of this access pattern
                l1, l2 = cp["divergent_64KB"], cp["divergent_4MB"]
                roof.update({"bound": "l1", "peak": l1, "frac": ach / l1, "frac_of_l2_resident_peak": ach / l2,
                             "peak_source": "measured live on this GPU by tools/peaks_cache: divergent 4 x 256-bit loads per 128-byte record, one "
                                            "record per lane, table resident in L1 (64 KB); l2 = same pattern over a 4 MB table",
                             "cache_peaks": cp})
            else:
                roof.update({"bound": "l1", "peak": None, "frac": None,
                             "peak_source": "tools/peaks_cache binary missing (run __graft_entry__.build())"})
        else:
            roof.update({"bound": "hbm", "achieved": hbm_def["achieved"], "peak": hbm_peak, "unit": "GB/s", "frac": hbm_def["frac"], "peak_source": how})
        roof["traffic"] = traffic.get("extend_dram_bytes_per_launch")
        if traffic.get("whole_step_dram_bytes"):
            rays_step = traffic.get("whole_step_rays") or (rays_all / args.steps)
            roof["dram"] = {"bytes_per_ray_whole_step": traffic["whole_step_dram_bytes"] / rays_step, "budget_bytes_per_ray": 64,
                            "whole_step_dram_bytes": traffic["whole_step_dram_bytes"],
                            "whole_step_gbs": traffic["whole_step_dram_bytes"] / (t_all / args.steps * 1e-3) / 1e9 if world == 1 else None,
                            "hbm_peak": hbm_peak, "source": traffic.get("file"),
                            "note": "dram__bytes_read.sum + dram__bytes_write.sum of every launch of one step (ncu --set full, committed capture)"}
        if world == 1 and not args.no_cpu_baseline:
            cpu = cpu_baseline(desc)

    # ---- the id-exact bounce-0 kernel against f32 primitive tests, primary rays alone (same scene, max_depth 0)
    if rank == 0 and world == 1 and prec == FAST_F32 and not args.no_primary:
        d0 = scenes.WORKLOADS[args.workload]()
        d0.max_depth = 0
        s0 = Scene(d0, bvh=bvh, device=local_rank)
        i0 = CudaPixelIntegrator(s0, precision=FAST_F32, seed=1)
        primary = {"workload": "same scene and frame, max_depth 0: every closest-hit ray is a primary ray", "spp": 16}
        for label, flags in (("id_exact_hybrid", 0), ("f32_primitive_tests", _lib.SAMPLE_F32_PRIMARY)):
            best = None
            for _ in range(3):
                i0.SampleF32(16, flags=flags)
                if best is None or i0.stats["ms_extend"] < best["ms_extend"]:
                    best = dict(i0.stats)
            primary[label] = {"primary_mrays_s": best["closest_rays"] / best["ms_extend"] / 1e3, "ms_extend": best["ms_extend"],
                              "fixups": best["hybrid_fixups"]}
        primary["note"] = ("bounce 0 of every frame in this file uses the id-exact kernel (mfx_hybrid.cu): primary-hit ids and t equal the "
                           "oracle's bit for bit (tests/test_gpu_parity.py::test_fast_primary_is_bit_exact)")
        s0.close()

    # ---- BASELINE configs[2..4] at their stated size through the same path (device timed, one warm + one timed full-size step each)
    configs = None
    if not args.no_configs and prec == FAST_F32:
        configs = []
        for name, spp in (("c3_renault", 256), ("c4_spheres", 128), ("c5_soup", 64)):
            dbg("config", name)
            cdesc = scenes.WORKLOADS[name]()
            t0 = time.perf_counter()
            cbvh = Bvh.Build(cdesc.prims)
            dbg("config", name, "tree built")
            t_bvh = time.perf_counter() - t0
            csc = Scene(cdesc, bvh=cbvh, device=local_rank)
            csh = mdist.ShardedPixelIntegrator(csc, rank, world, precision=prec, seed=1, stripe=mdist.STRIPE)
            t0 = time.perf_counter()
            csh.Sample(1)                                        # builds the layouts (own SAH tree, hybrid tables), untimed
            t_first = time.perf_counter() - t0
            sync_all()
            dbg("config", name, "layouts built")
            timed_step(csh, spp)                                 # untimed: the path state of a full-size wave is allocated here
            sync_all()
            ms, st = timed_step(csh, spp)
            dbg("config", name, "timed")
            r_all, t_cfg = aggregate(st["closest_rays"] + st["shadow_rays"], ms)
            row = {"config": name, "prims": int(len(cdesc.prims)), "size": [cdesc.width, cdesc.height], "spp": spp, "max_depth": cdesc.max_depth,
                   "integrator": ["PathIntegrator", "NewPathTracer", "GetColor"][cdesc.integrator], "n_gpus": world,
                   "rays": r_all, "ms": t_cfg, "mrays_s": r_all / t_cfg / 1e3, "spp_per_s": spp / (t_cfg * 1e-3),
                   "rank0": {"extend_mrays_s": st["closest_rays"] / max(st["ms_extend"], 1e-9) / 1e3,
                             "shadow_mrays_s": st["shadow_rays"] / max(st["ms_shadow"], 1e-9) / 1e3, "launches": st["launches"],
                             "hybrid_fixups": st["hybrid_fixups"]},
                   "host_bvh_build_s": t_bvh, "first_call_s": t_first, "scene_bytes": csc.device_bytes() if rank == 0 else None}
            if name == "c5_soup" and rank == 0:
                tr = load_traffic().get("c5")
                if tr:      # the one config whose scene leaves L2: HBM roofline from the committed ncu capture
                    row["hbm"] = tr
            configs.append(row)
            del csh
            csc.close()
            sync_all()

    dbg("configs done")
    if rank == 0:
        launches = sum(s["launches"] for s in stats)
        line = {"metric": METRIC, "value": value, "unit": "Mrays/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
                "ms_per_step": t_all / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "f32" if prec == FAST_F32 else "f64", "data": "synthetic",
                "config": {"workload": WORKLOAD if args.workload == "c2_spot" else args.workload, "spp": args.spp,
                           "parallelism": f"column stripes of {mdist.STRIPE} px interleaved over {world} GPU(s), scene replicated, "
                                          "1 NCCL gather of the owned stripes per frame" if world > 1 else "1 GPU, whole frame",
                           "l2": "256 MB buffer written between timed iterations (L2 flush); path state (184 B/path, one wave = pixels x spp up to 128 Mi paths = 24.6 GB) exceeds L2, scene is L2 resident by nature",
                           "primary_rays": "id-exact (hybrid kernel: f32 boxes, f64 primitive tests)" if prec == FAST_F32 else "exact f64",
                           "rays_per_step": rays_all / args.steps, "paths_per_step": desc.width * desc.height * args.spp},
                "spp_per_s": args.spp * args.steps / (t_all * 1e-3), "wall_s_timed_region": wall,
                "e2e": e2e, "gpu_launches": int(launches), "clocks": clk, "roofline": roof, "cpu_baseline": cpu,
                "primary": primary, "configs": configs}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
