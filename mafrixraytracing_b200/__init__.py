"""mafrixraytracing_b200 -- host-side mirror of MafrixRender's path-tracing interface over
libmafrix_cuda (hand-written sm_100a kernels behind a C ABI, include/mafrix_cuda.h).

Only what the hot path needs lives here:
  csrc/        CUDA kernels + the C ABI (built in-tree into libmafrix_cuda.so)
  _lib.py      ctypes binding of every symbol in include/mafrix_cuda.h (fails loudly if absent)
  scene.py     PinholeCamera / Bvh / Scene / CudaPixelIntegrator / Film -- the reference's names; their multi-GPU
               counterparts MultiGpuPixelIntegrator / MultiGpuFilm
  scenes.py    the BASELINE workload builders (C1..C5) and the sphere sample's RandomScene
  imageio.py   headless PFM / PNG writers (replace the reference's ImGui window)
  dist.py      one-process-per-GPU sharding (torchrun): stripes per rank + the NCCL gather of the owned stripes
There is no CPU fallback: without the CUDA library or a GPU every compute call raises.
"""
from .scene import (PRIM_DTYPE, MATERIAL_DTYPE, NODE_DTYPE, TRIANGLE, RECT, SPHERE, LAMBERT, METAL,
                    SPECTRANS, DIELECTRIC, LAMBERT_CHECKER, LAMBERT_NOISE, PATH_INTEGRATOR, NEW_PATH_TRACER,
                    SKY_TRACER, EXACT_F64, FAST_F32,
                    PinholeCamera, RayTraceCamera, SkyTracer, AreaLight, SceneDesc, Bvh, Scene, CudaPixelIntegrator,
                    MultiGpuPixelIntegrator, Film, MultiGpuFilm, MafrixError)

__all__ = ["PRIM_DTYPE", "MATERIAL_DTYPE", "NODE_DTYPE", "TRIANGLE", "RECT", "SPHERE", "LAMBERT",
           "METAL", "SPECTRANS", "DIELECTRIC", "LAMBERT_CHECKER", "LAMBERT_NOISE", "PATH_INTEGRATOR",
           "NEW_PATH_TRACER", "SKY_TRACER", "EXACT_F64", "FAST_F32",
           "PinholeCamera", "RayTraceCamera", "SkyTracer", "AreaLight", "SceneDesc", "Bvh", "Scene", "CudaPixelIntegrator",
           "MultiGpuPixelIntegrator", "Film", "MultiGpuFilm", "MafrixError"]
