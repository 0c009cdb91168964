"""Host-side mirror of the reference's path-tracing interface, over the C ABI.

Names and argument meaning follow the F# types they stand in for (paths under
/root/reference/EngineCore/):

  PinholeCamera(pos, dir, fov, aspect)        Core/Camera.fs:113-142
  AreaLight(p0,p1,p2,p3, normal, color)       Core/Lights/Light.fs:32-64 (NewAreaLight)
  Bvh.Build(prims)                            Core/Accelerate/BvhNode.fs:24-30
  Scene(desc) / Scene.Hit / TracePrimary      Scene/Scene.fs:298-313, BvhNode.fs:83
  CudaPixelIntegrator.Sample(n)               Core/Integrator/Integrators.fs:143-172 (IPixelIntegrator)
  Film.GetFrame(integrator, samples)          Core/Film.fs:13-34
  RayTraceCamera(lookfrom, lookat, vup, ...)  RenderTest/Sample/RayTracing.fs:335-364 (the sphere sample, SKY_TRACER)

All compute goes through libmafrix_cuda; nothing here renders on the CPU.
"""
import ctypes as C
import weakref
from dataclasses import dataclass, field

import numpy as np

from . import _lib
from ._lib import MafrixError  # noqa: F401  (re-exported)

# MfxPrim / MfxMaterial / MfxBvhNode (include/mafrix_cuda.h)
PRIM_DTYPE = np.dtype([("kind", "<i4"), ("material", "<i4"), ("v", "<f8", (12,))])
MATERIAL_DTYPE = np.dtype([("kind", "<i4"), ("pad", "<i4"), ("albedo", "<f8", (3,)),
                           ("fuzz", "<f8"), ("ei", "<f8"), ("et", "<f8")])
NODE_DTYPE = np.dtype([("pmin", "<f8", (3,)), ("pmax", "<f8", (3,)), ("first", "<i4"), ("count", "<i4")])
assert PRIM_DTYPE.itemsize == 104 and MATERIAL_DTYPE.itemsize == 56 and NODE_DTYPE.itemsize == 56

TRIANGLE, RECT, SPHERE = 0, 1, 2
LAMBERT, METAL, SPECTRANS = 0, 1, 2
DIELECTRIC, LAMBERT_CHECKER, LAMBERT_NOISE = 3, 4, 5      # SKY_TRACER only (RayTracing.fs:300-325, :54-61, :96-99)
PATH_INTEGRATOR, NEW_PATH_TRACER, SKY_TRACER = 0, 1, 2
EXACT_F64, FAST_F32 = 0, 1


def _vec3(x):
    a = np.ascontiguousarray(x, dtype=np.float64).reshape(3)
    return a


class PinholeCamera:
    """PinholeCamera(pos, dir, fov, aspectRatio): derived on the host exactly like Camera.fs:96-133
    (effective FOV = fov/2, `right` not re-normalised)."""

    def __init__(self, pos, dir, fov, aspect):
        self.pos_arg, self.dir_arg = _vec3(pos), _vec3(dir)
        self.fov, self.aspect = float(fov), float(aspect)
        cam = _lib.MfxCamera()
        _lib.check(_lib.load().mfx_camera_pinhole(_lib.ptr(self.pos_arg), _lib.ptr(self.dir_arg), self.fov,
                                                  self.aspect, C.byref(cam)))
        self._c = cam
        self.position = np.array(cam.pos[:])
        self.topleft = np.array(cam.topleft[:])
        self.right = np.array(cam.right[:])
        self.down = np.array(cam.down[:])

    def derived(self):
        """pos, topleft, right, down as one (12,) f64 array."""
        return np.concatenate([self.position, self.topleft, self.right, self.down])

    def GetRay(self, u, v):
        """Camera.fs:134-139 (host convenience for tests; the kernels generate their own rays)."""
        target = (self.topleft + u * self.right) + v * self.down
        d = target - self.position
        l = np.sqrt(d[0] * d[0] + d[1] * d[1] + d[2] * d[2])
        return self.position.copy(), d / l


class RayTraceCamera:
    """RayTraceCamera(lookfrom, lookat, vup, vfov, aspect, aperture, focus_dist, t0, t1) of the sphere sample
    (RenderTest/Sample/RayTracing.fs:335-358), derived on the host by the library; t0/t1 only feed MovingSphere,
    which is not carried over."""

    def __init__(self, lookfrom, lookat, vup, vfov, aspect, aperture=0.0, focus_dist=None):
        self.lookfrom, self.lookat, self.vup = _vec3(lookfrom), _vec3(lookat), _vec3(vup)
        self.vfov, self.aspect, self.aperture = float(vfov), float(aspect), float(aperture)
        if focus_dist is None:                                   # dist_to_focus = (lookfrom-lookat).Length, :431
            d = self.lookfrom - self.lookat
            focus_dist = np.sqrt(d[0] * d[0] + d[1] * d[1] + d[2] * d[2])
        self.focus_dist = float(focus_dist)
        cam = _lib.MfxLensCamera()
        _lib.check(_lib.load().mfx_camera_lens(_lib.ptr(self.lookfrom), _lib.ptr(self.lookat), _lib.ptr(self.vup),
                                               self.vfov, self.aspect, self.aperture, self.focus_dist, C.byref(cam)))
        self._c = cam

    def derived(self):
        """origin, lower_left, horizontal, vertical, u, v, lens_radius as one (19,) f64 array."""
        c = self._c
        return np.array(list(c.origin) + list(c.lower_left) + list(c.horizontal) + list(c.vertical) + list(c.u) +
                        list(c.v) + [c.lens_radius])


@dataclass
class SkyTracer:
    """What the sphere sample needs beyond shapes and materials: its camera and Perlin's static tables
    (RayTracing.fs:81-85; ranfloat[256], perm = perm_x|perm_y|perm_z [3*256]; None without a noise material)."""
    camera: RayTraceCamera
    ranfloat: np.ndarray = None
    perm: np.ndarray = None

    def __post_init__(self):
        if self.ranfloat is not None:
            self.ranfloat = np.ascontiguousarray(self.ranfloat, dtype=np.float64).reshape(256)
        if self.perm is not None:
            self.perm = np.ascontiguousarray(self.perm, dtype=np.int32).reshape(768)


@dataclass
class AreaLight:
    """NewAreaLight(p0,p1,p2,p3,nm,c) (Light.fs:36-41)."""
    p: np.ndarray          # (4,3)
    normal: np.ndarray     # (3,)
    color: np.ndarray      # (3,)

    def __post_init__(self):
        self.p = np.ascontiguousarray(self.p, dtype=np.float64).reshape(4, 3)
        self.normal = _vec3(self.normal)
        self.color = _vec3(self.color)


def make_prims(n):
    return np.zeros(n, dtype=PRIM_DTYPE)


def triangles_from_mesh(v, f, material=0):
    """ObjModelLoader.Face.ToHitable (ObjModelLoader.fs:63-92): 3 vertices -> Triangle, 4 -> Rect."""
    v = np.asarray(v, np.float64)
    f = np.asarray(f, np.int32)
    prims = make_prims(len(f))
    quad = f[:, 3] >= 0
    prims["kind"] = np.where(quad, RECT, TRIANGLE)
    prims["material"] = material
    pv = prims["v"]
    pv[:, 0:3] = v[f[:, 0]]
    pv[:, 3:6] = v[f[:, 1]]
    pv[:, 6:9] = v[f[:, 2]]
    pv[quad, 9:12] = v[f[quad, 3]]
    return prims


def rect_prim(p0, p1, p2, p3, material=0):
    r = make_prims(1)
    r["kind"] = RECT
    r["material"] = material
    r["v"][0] = np.concatenate([_vec3(p0), _vec3(p1), _vec3(p2), _vec3(p3)])
    return r


def sphere_prims(centers, radii, materials):
    centers = np.asarray(centers, np.float64).reshape(-1, 3)
    s = make_prims(len(centers))
    s["kind"] = SPHERE
    s["material"] = materials
    s["v"][:, 0:3] = centers
    s["v"][:, 3] = radii
    return s


def make_materials(specs):
    """specs: list of ("lambert", (r,g,b)) | ("metal", (r,g,b), fuzz) | ("spectrans", (r,g,b), ei, et); SKY_TRACER
    adds ("dielectric", ri) | ("checker", even_rgb, odd_rgb) | ("noise",)."""
    m = np.zeros(len(specs), dtype=MATERIAL_DTYPE)
    for i, s in enumerate(specs):
        kind = {"lambert": LAMBERT, "metal": METAL, "spectrans": SPECTRANS, "dielectric": DIELECTRIC,
                "checker": LAMBERT_CHECKER, "noise": LAMBERT_NOISE}[s[0]]
        m[i]["kind"] = kind
        if kind == DIELECTRIC:
            m[i]["albedo"] = (1., 1., 1.)
            m[i]["ei"] = s[1]
            continue
        if kind == LAMBERT_NOISE:
            m[i]["albedo"] = (1., 1., 1.)
            continue
        m[i]["albedo"] = s[1]
        if kind == METAL:
            m[i]["fuzz"] = s[2]
        if kind == SPECTRANS:
            m[i]["ei"], m[i]["et"] = s[2], s[3]
        if kind == LAMBERT_CHECKER:                      # odd colour rides in (fuzz, ei, et), see MfxMaterial
            m[i]["fuzz"], m[i]["ei"], m[i]["et"] = s[2]
    return m


@dataclass
class SceneDesc:
    """What `new Scene(state)` consumes (Scene.fs:298-313): shapes, the resolved material table,
    the area light, the camera, the film size, maxDepth and which IPathTracer runs."""
    prims: np.ndarray
    materials: np.ndarray
    light: AreaLight
    camera: PinholeCamera
    width: int
    height: int
    max_depth: int = 3                  # Scene.fs:304
    integrator: int = PATH_INTEGRATOR
    name: str = ""
    meta: dict = field(default_factory=dict)
    sky: SkyTracer = None               # SKY_TRACER: light and camera are ignored (pass None)

    def __post_init__(self):
        self.prims = np.ascontiguousarray(self.prims, dtype=PRIM_DTYPE)
        self.materials = np.ascontiguousarray(self.materials, dtype=MATERIAL_DTYPE)


class Bvh:
    """Bvh.Build (BvhNode.fs:24-61) reproduced on the host by the library (mfx_bvh_build)."""

    def __init__(self, nodes, indices):
        self.nodes = np.ascontiguousarray(nodes, dtype=NODE_DTYPE)
        self.indices = np.ascontiguousarray(indices, dtype=np.int32)

    @staticmethod
    def Build(prims):
        prims = np.ascontiguousarray(prims, dtype=PRIM_DTYPE)
        n = len(prims)
        nodes = np.zeros(2 * n - 1, dtype=NODE_DTYPE)
        indices = np.zeros(n, dtype=np.int32)
        _lib.check(_lib.load().mfx_bvh_build(_lib.ptr(prims), n, _lib.ptr(nodes), len(nodes), _lib.ptr(indices)))
        return Bvh(nodes, indices)


class Scene:
    """The device-resident scene: flattened tree + primitives + materials + light + camera."""

    def __init__(self, desc: SceneDesc, bvh: Bvh = None, device: int = None):
        lib = _lib.load()
        if device is not None:
            _lib.check(lib.mfx_init(int(device)))
        self.desc = desc
        self.width, self.height = int(desc.width), int(desc.height)
        d = self._c_desc(desc, bvh)
        h = C.c_void_p()
        _lib.check(lib.mfx_scene_create(C.byref(d), C.byref(h)))
        self._h = h
        self._films = weakref.WeakSet()

    def _c_desc(self, desc, bvh):
        """MfxSceneDesc over the arrays of `desc` (kept alive by it) -- what `new Scene(state)` consumes."""
        d = _lib.MfxSceneDesc()
        d.prims = _lib.ptr(desc.prims)
        d.n_prims = len(desc.prims)
        d.materials = _lib.ptr(desc.materials)
        d.n_materials = len(desc.materials)
        if bvh is not None:
            d.nodes = _lib.ptr(bvh.nodes)
            d.n_node_slots = len(bvh.nodes)
            d.indices = _lib.ptr(bvh.indices)
        else:
            d.nodes, d.n_node_slots, d.indices = None, 0, None
        if desc.light is not None:
            d.light.p[:] = desc.light.p.reshape(-1).tolist()
            d.light.normal[:] = desc.light.normal.tolist()
            d.light.color[:] = desc.light.color.tolist()
        if desc.camera is not None:
            d.camera = desc.camera._c
        if desc.sky is not None:
            self._sky = _lib.MfxSkyTracer()
            self._sky.camera = desc.sky.camera._c
            self._sky.perlin_ranfloat = _lib.ptr(desc.sky.ranfloat)
            self._sky.perlin_perm = _lib.ptr(desc.sky.perm)
            d.sky = C.pointer(self._sky)
        d.width, d.height = int(desc.width), int(desc.height)
        d.max_depth, d.integrator = int(desc.max_depth), int(desc.integrator)
        self._bvh_keep = bvh
        return d

    def close(self):
        if getattr(self, "_h", None):
            for f in list(getattr(self, "_films", ())):      # a Film borrows the scene's stream and buffers: it goes first
                f.close()
            _lib.load().mfx_scene_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def Prepare(self, precision=FAST_F32):
        """Builds the device layouts of `precision` now instead of inside the first Sample."""
        _lib.check(_lib.load().mfx_scene_prepare(self._h, int(precision)))

    def bvh(self):
        n = len(self.desc.prims)
        nodes = np.zeros(2 * n - 1, dtype=NODE_DTYPE)
        indices = np.zeros(n, dtype=np.int32)
        _lib.check(_lib.load().mfx_scene_get_bvh(self._h, _lib.ptr(nodes), _lib.ptr(indices)))
        return Bvh(nodes, indices)

    def device_bytes(self):
        a, b = C.c_uint64(), C.c_uint64()
        _lib.check(_lib.load().mfx_scene_device_bytes(self._h, C.byref(a), C.byref(b)))
        return {"exact": a.value, "fast": b.value}

    def Hit(self, origins, dirs, tmin, tmax, precision=EXACT_F64, any_hit=False):
        """Bvh.Hit(ray, tMin, tMax) for n rays -> (prim, sub, t)."""
        o = np.ascontiguousarray(origins, np.float64).reshape(-1, 3)
        d = np.ascontiguousarray(dirs, np.float64).reshape(-1, 3)
        n = len(o)
        prim = np.full(n, -1, np.int32)
        sub = np.zeros(n, np.int32)
        t = np.zeros(n, np.float64)
        _lib.check(_lib.load().mfx_bvh_hit(self._h, precision, int(any_hit), n, _lib.ptr(o), _lib.ptr(d),
                                           float(tmin), float(tmax), _lib.ptr(prim), _lib.ptr(sub), _lib.ptr(t)))
        return prim, sub, t

    def HitFrom(self, origins, dirs, src, tmin, tmax, any_hit=False):
        """Bvh.Hit for n rays that start on primitive src[i] (-1: none; None: none at all), traced by the f32 kernel of
        bounces >= 1 and shadow rays -> (prim, sub, t)."""
        o = np.ascontiguousarray(origins, np.float64).reshape(-1, 3)
        d = np.ascontiguousarray(dirs, np.float64).reshape(-1, 3)
        n = len(o)
        sp = None if src is None else np.ascontiguousarray(src, np.int32).reshape(n)
        prim = np.full(n, -1, np.int32)
        sub = np.zeros(n, np.int32)
        t = np.zeros(n, np.float64)
        _lib.check(_lib.load().mfx_bvh_hit_from(self._h, int(any_hit), n, _lib.ptr(o), _lib.ptr(d),
                                                None if sp is None else _lib.ptr(sp), float(tmin), float(tmax),
                                                _lib.ptr(prim), _lib.ptr(sub), _lib.ptr(t)))
        return prim, sub, t

    def TracePrimary(self, uv=None, precision=EXACT_F64):
        """cam.GetRay(u,v) + bvh.Hit(ray,1e-6,99999999.) -> (prim, t); uv None = pixel centres (row-major)."""
        if uv is None:
            n = self.width * self.height
            uvp = None
        else:
            uv = np.ascontiguousarray(uv, np.float64).reshape(-1, 2)
            n = len(uv)
            uvp = _lib.ptr(uv)
        prim = np.full(n, -1, np.int32)
        t = np.zeros(n, np.float64)
        _lib.check(_lib.load().mfx_trace_primary(self._h, precision, n, uvp, _lib.ptr(prim), _lib.ptr(t)))
        return prim, t


class CudaPixelIntegrator:
    """IPixelIntegrator over the GPU: Sample(n) returns the reference's Texture2D<Color> as a
    (width, height, 4) f64 array -- element [x, y] = Color(r, g, b, 1)."""

    def __init__(self, scene: Scene, precision=FAST_F32, seed=1, tile_size=0, rank=0, world=1):
        self.scene = scene
        self.precision, self.seed = int(precision), int(seed)
        self.tile_size, self.rank, self.world = int(tile_size), int(rank), int(world)
        self.texture = np.zeros((scene.width, scene.height, 4), dtype=np.float64)
        self.stats = None

    def _params(self, n, first_sample, flags=0):
        return _lib.MfxSampleParams(self.precision, int(n), self.seed, int(first_sample), self.tile_size,
                                    self.rank, self.world, int(flags))

    def _after(self):
        st = _lib.MfxStats()
        _lib.check(_lib.load().mfx_get_stats(self.scene._h, C.byref(st)))
        self.stats = {k: (list(getattr(st, k)) if k in ("nodes", "tris", "spheres") else getattr(st, k))
                      for k, _ in _lib.MfxStats._fields_ if k != "pad"}

    def Sample(self, n, first_sample=0, flags=0, out=None):
        tex = self.texture if out is None else out
        p = self._params(n, first_sample, flags)
        _lib.check(_lib.load().mfx_pixel_integrator_sample(self.scene._h, C.byref(p), _lib.ptr(tex)))
        self._after()
        return tex

    def SampleAsync(self, n, out, first_sample=0, flags=0):
        """Enqueues Sample(n) into the PINNED texture `out` (mfx_host_register) and returns; Wait() completes the oldest
        frame in flight (two at most: frame k downloads while frame k+1 renders)."""
        p = self._params(n, first_sample, flags)
        _lib.check(_lib.load().mfx_pixel_integrator_sample_async(self.scene._h, C.byref(p), _lib.ptr(out)))

    def Wait(self):
        _lib.check(_lib.load().mfx_pixel_integrator_wait(self.scene._h))
        self._after()

    def SampleF32(self, n, first_sample=0, flags=0):
        """Row-major (height, width, 4) float32 image (PFM/PNG writers)."""
        img = np.zeros((self.scene.height, self.scene.width, 4), dtype=np.float32)
        p = self._params(n, first_sample, flags)
        _lib.check(_lib.load().mfx_pixel_integrator_sample_f32(self.scene._h, C.byref(p), _lib.ptr(img)))
        self._after()
        return img

    def SampleDevice(self, n, device_ptr, first_sample=0, flags=0):
        """Leaves the (height*width) float4 frame in caller-owned device memory (e.g. a torch
        tensor's data_ptr()) so the multi-GPU reduce runs on it without a host round trip."""
        p = self._params(n, first_sample, flags)
        _lib.check(_lib.load().mfx_pixel_integrator_sample_device(self.scene._h, C.byref(p), C.c_void_p(int(device_ptr))))
        self._after()


    def SampleDeviceColor(self, n, device_ptr, first_sample=0, flags=0):
        """Leaves Color[w,h] (width*height*4 f64, x-major: the reference's Texture2D layout) in caller-owned device memory."""
        p = self._params(n, first_sample, flags)
        _lib.check(_lib.load().mfx_pixel_integrator_sample_device_color(self.scene._h, C.byref(p), C.c_void_p(int(device_ptr))))
        self._after()


class MultiGpuPixelIntegrator:
    """IPixelIntegrator over several GPUs behind ONE host thread (mfx_multi_*): the scene is replicated on every device,
    the library shards the frame by column stripes and every device writes its stripes straight into `texture`."""

    def __init__(self, desc: SceneDesc, devices=None, n_devices=0, bvh: Bvh = None, precision=FAST_F32, seed=1):
        self._keep = Scene.__new__(Scene)                    # borrow Scene's descriptor marshalling without creating a scene
        lib = _lib.load()
        self.desc, self.precision, self.seed = desc, int(precision), int(seed)
        self.width, self.height = int(desc.width), int(desc.height)
        d = Scene._c_desc(self._keep, desc, bvh)
        devs = None if devices is None else np.ascontiguousarray(devices, dtype=np.int32)
        h = C.c_void_p()
        _lib.check(lib.mfx_multi_create(C.byref(d), _lib.ptr(devs), len(devs) if devs is not None else int(n_devices), C.byref(h)))
        self._h = h
        n = C.c_int32()
        _lib.check(lib.mfx_multi_device_count(self._h, C.byref(n)))
        self.n_devices = n.value
        self.texture = np.zeros((self.width, self.height, 4), dtype=np.float64)
        self.stats = None
        self._films = weakref.WeakSet()

    def close(self):
        if getattr(self, "_h", None):
            for f in list(getattr(self, "_films", ())):      # mfx_multi_destroy refuses while a film of the handle lives
                f.close()
            _lib.load().mfx_multi_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _after(self):
        st = _lib.MfxStats()
        per = (_lib.MfxStats * self.n_devices)()
        _lib.check(_lib.load().mfx_multi_get_stats(self._h, C.byref(st), C.cast(per, C.c_void_p)))
        conv = lambda x: {k: (list(getattr(x, k)) if k in ("nodes", "tris", "spheres") else getattr(x, k)) for k, _ in _lib.MfxStats._fields_}
        self.stats = conv(st)
        self.stats["per_device"] = [conv(x) for x in per]

    def Sample(self, n, first_sample=0, flags=0, out=None):
        tex = self.texture if out is None else out
        p = _lib.MfxSampleParams(self.precision, int(n), self.seed, int(first_sample), 0, 0, 1, int(flags))
        _lib.check(_lib.load().mfx_multi_sample(self._h, C.byref(p), _lib.ptr(tex)))
        self._after()
        return tex

    def Prepare(self):
        """Builds every replica's device layouts now instead of inside the first Sample."""
        _lib.check(_lib.load().mfx_multi_prepare(self._h, self.precision))

    def SampleAsync(self, n, out, first_sample=0, flags=0):
        """Posts Sample(n) to the device workers and returns; Wait() completes it (one frame in flight per handle)."""
        p = _lib.MfxSampleParams(self.precision, int(n), self.seed, int(first_sample), 0, 0, 1, int(flags))
        _lib.check(_lib.load().mfx_multi_sample_async(self._h, C.byref(p), _lib.ptr(out)))

    def Wait(self):
        _lib.check(_lib.load().mfx_multi_wait(self._h))
        self._after()

    def SampleF32(self, n, first_sample=0, flags=0):
        img = np.zeros((self.height, self.width, 4), dtype=np.float32)
        p = _lib.MfxSampleParams(self.precision, int(n), self.seed, int(first_sample), 0, 0, 1, int(flags))
        _lib.check(_lib.load().mfx_multi_sample_f32(self._h, C.byref(p), _lib.ptr(img)))
        self._after()
        return img


class _FilmBase:
    """What Film and MultiGpuFilm share: sum += frame; target = sum / frameCount, kept in HBM.  `_c` is the prefix of the
    subclass's C functions; `owner` is the Scene or MultiGpuPixelIntegrator the film lives on, whose close() closes the
    film first."""

    _c = None

    def __init__(self, owner):
        self._owner = owner
        h = C.c_void_p()
        _lib.check(self._fn("create")(owner._h, C.byref(h)))
        self._h = h
        owner._films.add(self)
        self.target = np.zeros((owner.width, owner.height, 4), dtype=np.float64)

    def _fn(self, name):
        return getattr(_lib.load(), f"{self._c}_{name}")

    def close(self):
        if getattr(self, "_h", None):
            self._fn("destroy")(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def Reset(self):
        _lib.check(self._fn("reset")(self._h))

    def FrameCount(self):
        fc = C.c_double()
        _lib.check(self._fn("frame_count")(self._h, C.byref(fc)))
        return fc.value

    def Export(self):
        """Checkpoint: (running sum Color[w,h], frameCount) -- all the state Film carries (Film.fs:14-17)."""
        s = np.zeros((self._owner.width, self._owner.height, 4), dtype=np.float64)
        fc = C.c_double()
        _lib.check(self._fn("export")(self._h, _lib.ptr(s), C.byref(fc)))
        return s, fc.value

    def Import(self, sum_wh, frame_count):
        sum_wh = np.ascontiguousarray(sum_wh, dtype=np.float64)
        want = (self._owner.width, self._owner.height, 4)
        if sum_wh.shape != want:
            raise ValueError(f"{type(self).__name__}.Import: running sum has shape {sum_wh.shape}, the film is Color[w,h] = {want}")
        _lib.check(self._fn("import")(self._h, _lib.ptr(sum_wh), float(frame_count)))

    def PostProcess(self, out=None):
        """Scene.PostProcessAndToScreenBuffer (Scene.fs:315-330) -> (height, width, 4) uint8."""
        if out is None:
            out = np.zeros((self._owner.height, self._owner.width, 4), dtype=np.uint8)
        _lib.check(self._fn("post_process")(self._h, _lib.ptr(out)))
        return out


class Film(_FilmBase):
    """Film (Film.fs:13-34) on one GPU."""

    _c = "mfx_film"

    def __init__(self, scene: Scene):
        self.scene = scene
        super().__init__(scene)

    def GetFrame(self, integrator: CudaPixelIntegrator, samples, first_sample=None):
        if first_sample is None:
            first_sample = int(self.FrameCount()) * int(samples)     # fresh samples every frame
        p = integrator._params(samples, first_sample)
        _lib.check(_lib.load().mfx_film_get_frame(self._h, C.byref(p), _lib.ptr(self.target)))
        integrator._after()
        return self.target


class MultiGpuFilm(_FilmBase):
    """Film over several GPUs (mfx_multi_film_*): every device of `multi` accumulates, divides and tone-maps its own
    column stripes in its own HBM.  Same surface and the same results, bit for bit, as Film on one GPU."""

    _c = "mfx_multi_film"

    def __init__(self, multi: MultiGpuPixelIntegrator):
        self.multi = multi
        super().__init__(multi)

    def GetFrame(self, samples, first_sample=None, download=True):
        """Film.GetFrame over every device -> target as Color[w,h]; download=False keeps it on the devices (a host that
        only displays calls PostProcess next) and returns None."""
        if first_sample is None:
            first_sample = int(self.FrameCount()) * int(samples)     # fresh samples every frame
        m = self.multi
        p = _lib.MfxSampleParams(m.precision, int(samples), m.seed, int(first_sample), 0, 0, 1, 0)
        _lib.check(_lib.load().mfx_multi_film_get_frame(self._h, C.byref(p), _lib.ptr(self.target) if download else None))
        m._after()
        return self.target if download else None
