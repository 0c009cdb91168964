"""ctypes binding of libmafrix_cuda.so (include/mafrix_cuda.h).  No fallback of any kind:
if the library is missing this module raises, and every compute entry point returns
MFX_ERR_NO_DEVICE (raised as MafrixError) when no GPU is visible."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# MFX_LIB: another build of the same ABI (the `make DEBUG=1` flavour with bounds checks, libmafrix_cuda_dbg.so)
LIB_PATH = os.environ.get("MFX_LIB") or os.path.join(_HERE, "libmafrix_cuda.so")


class MafrixError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libmafrix_cuda error {code}: {msg}")
        self.code = code


class MfxAreaLight(C.Structure):
    _fields_ = [("p", C.c_double * 12), ("normal", C.c_double * 3), ("color", C.c_double * 3)]


class MfxCamera(C.Structure):
    _fields_ = [("pos", C.c_double * 3), ("topleft", C.c_double * 3), ("right", C.c_double * 3),
                ("down", C.c_double * 3)]


class MfxLensCamera(C.Structure):
    _fields_ = [("origin", C.c_double * 3), ("lower_left", C.c_double * 3), ("horizontal", C.c_double * 3),
                ("vertical", C.c_double * 3), ("u", C.c_double * 3), ("v", C.c_double * 3),
                ("lens_radius", C.c_double)]


class MfxSkyTracer(C.Structure):
    _fields_ = [("camera", MfxLensCamera), ("perlin_ranfloat", C.c_void_p), ("perlin_perm", C.c_void_p)]


class MfxSceneDesc(C.Structure):
    _fields_ = [("prims", C.c_void_p), ("n_prims", C.c_int32),
                ("materials", C.c_void_p), ("n_materials", C.c_int32),
                ("nodes", C.c_void_p), ("n_node_slots", C.c_int32),
                ("indices", C.c_void_p),
                ("light", MfxAreaLight), ("camera", MfxCamera),
                ("width", C.c_int32), ("height", C.c_int32),
                ("max_depth", C.c_int32), ("integrator", C.c_int32),
                ("sky", C.POINTER(MfxSkyTracer))]


class MfxSampleParams(C.Structure):
    _fields_ = [("precision", C.c_int32), ("spp", C.c_int32), ("seed", C.c_uint64),
                ("first_sample", C.c_int32), ("tile_size", C.c_int32),
                ("rank", C.c_int32), ("world", C.c_int32), ("flags", C.c_int32)]


class MfxStats(C.Structure):
    _fields_ = [("closest_rays", C.c_uint64), ("shadow_rays", C.c_uint64), ("paths", C.c_uint64),
                ("nodes", C.c_uint64 * 2), ("tris", C.c_uint64 * 2), ("spheres", C.c_uint64 * 2),
                ("ms_total", C.c_double), ("ms_extend", C.c_double), ("ms_shadow", C.c_double),
                ("ms_shade", C.c_double),
                ("launches", C.c_uint32), ("launches_extend", C.c_uint32),
                ("launches_shadow", C.c_uint32), ("hybrid_fixups", C.c_uint32)]


SAMPLE_COUNT_TRAVERSAL = 1
SAMPLE_REFERENCE_STREAM = 2
SAMPLE_COUNT_OWN_TREE = 4
SAMPLE_F32_PRIMARY = 8
SAMPLE_STRIPES = 16
SAMPLE_NO_CLEAR = 32

# every symbol include/mafrix_cuda.h declares: name -> (restype, argtypes)
_P = C.c_void_p
SYMBOLS = {
    "mfx_version": (C.c_char_p, []),
    "mfx_last_error": (C.c_char_p, []),
    "mfx_device_count": (C.c_int, []),
    "mfx_init": (C.c_int, [C.c_int]),
    "mfx_camera_pinhole": (C.c_int, [_P, _P, C.c_double, C.c_double, C.POINTER(MfxCamera)]),
    "mfx_camera_lens": (C.c_int, [_P, _P, _P, C.c_double, C.c_double, C.c_double, C.c_double, C.POINTER(MfxLensCamera)]),
    "mfx_bvh_build": (C.c_int, [_P, C.c_int32, _P, C.c_int32, _P]),
    "mfx_tile_map": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _P, C.POINTER(C.c_int32)]),
    "mfx_stripe_map": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _P, C.POINTER(C.c_int32)]),
    "mfx_scene_create": (C.c_int, [C.POINTER(MfxSceneDesc), C.POINTER(_P)]),
    "mfx_scene_destroy": (C.c_int, [_P]),
    "mfx_scene_prepare": (C.c_int, [_P, C.c_int32]),
    "mfx_scene_get_bvh": (C.c_int, [_P, _P, _P]),
    "mfx_scene_device_bytes": (C.c_int, [_P, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
    "mfx_bvh_hit": (C.c_int, [_P, C.c_int32, C.c_int32, C.c_int64, _P, _P, C.c_double, C.c_double, _P, _P, _P]),
    "mfx_bvh_hit_from": (C.c_int, [_P, C.c_int32, C.c_int64, _P, _P, _P, C.c_double, C.c_double, _P, _P, _P]),
    "mfx_trace_primary": (C.c_int, [_P, C.c_int32, C.c_int64, _P, _P, _P]),
    "mfx_pixel_integrator_sample": (C.c_int, [_P, C.POINTER(MfxSampleParams), _P]),
    "mfx_pixel_integrator_sample_async": (C.c_int, [_P, C.POINTER(MfxSampleParams), _P]),
    "mfx_pixel_integrator_wait": (C.c_int, [_P]),
    "mfx_pixel_integrator_sample_device": (C.c_int, [_P, C.POINTER(MfxSampleParams), _P]),
    "mfx_pixel_integrator_sample_device_color": (C.c_int, [_P, C.POINTER(MfxSampleParams), _P]),
    "mfx_pixel_integrator_sample_f32": (C.c_int, [_P, C.POINTER(MfxSampleParams), _P]),
    "mfx_get_stats": (C.c_int, [_P, C.POINTER(MfxStats)]),
    "mfx_host_register": (C.c_int, [_P, C.c_uint64]),
    "mfx_host_unregister": (C.c_int, [_P]),
    "mfx_multi_create": (C.c_int, [C.POINTER(MfxSceneDesc), _P, C.c_int32, C.POINTER(_P)]),
    "mfx_multi_destroy": (C.c_int, [_P]),
    "mfx_multi_device_count": (C.c_int, [_P, C.POINTER(C.c_int32)]),
    "mfx_multi_sample": (C.c_int, [_P, C.POINTER(MfxSampleParams), _P]),
    "mfx_multi_sample_async": (C.c_int, [_P, C.POINTER(MfxSampleParams), _P]),
    "mfx_multi_wait": (C.c_int, [_P]),
    "mfx_multi_prepare": (C.c_int, [_P, C.c_int32]),
    "mfx_multi_sample_f32": (C.c_int, [_P, C.POINTER(MfxSampleParams), _P]),
    "mfx_multi_get_stats": (C.c_int, [_P, C.POINTER(MfxStats), _P]),
    "mfx_film_create": (C.c_int, [_P, C.POINTER(_P)]),
    "mfx_film_destroy": (C.c_int, [_P]),
    "mfx_film_reset": (C.c_int, [_P]),
    "mfx_film_get_frame": (C.c_int, [_P, C.POINTER(MfxSampleParams), _P]),
    "mfx_film_post_process": (C.c_int, [_P, _P]),
    "mfx_film_frame_count": (C.c_int, [_P, C.POINTER(C.c_double)]),
    "mfx_film_export": (C.c_int, [_P, _P, C.POINTER(C.c_double)]),
    "mfx_film_import": (C.c_int, [_P, _P, C.c_double]),
    "mfx_multi_film_create": (C.c_int, [_P, C.POINTER(_P)]),
    "mfx_multi_film_destroy": (C.c_int, [_P]),
    "mfx_multi_film_reset": (C.c_int, [_P]),
    "mfx_multi_film_get_frame": (C.c_int, [_P, C.POINTER(MfxSampleParams), _P]),
    "mfx_multi_film_post_process": (C.c_int, [_P, _P]),
    "mfx_multi_film_frame_count": (C.c_int, [_P, C.POINTER(C.c_double)]),
    "mfx_multi_film_export": (C.c_int, [_P, _P, C.POINTER(C.c_double)]),
    "mfx_multi_film_import": (C.c_int, [_P, _P, C.c_double]),
}

_lib = None


def load():
    """Loads libmafrix_cuda.so (built by __graft_entry__.build() / csrc/Makefile)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                              "(there is no CPU fallback)")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(lib, name)          # AttributeError if the symbol is not exported
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def check(rc):
    if rc != 0:
        raise MafrixError(rc, load().mfx_last_error().decode("utf-8", "replace"))


def ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)
