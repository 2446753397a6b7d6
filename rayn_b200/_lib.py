"""ctypes binding of the C ABI in include/rayn_b200.h.

The product path has NO CPU fallback: if the CUDA library is missing this module raises at
import of the symbol table, and `rayn_b200_create` fails with RAYN_ERR_NO_DEVICE on a box
without a GPU.  Nothing here imports or touches oracle/.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# Which build of the library: RAYN_MULADD_FUSED=1 selects the variant with `wide` mul_add fused (oracle/README.md A6);
# RAYN_B200_LEGACY=1 the TEST build that also carries the round-1 one-thread-per-ray kernels.  Default = the product.
MULADD_FUSED = os.environ.get("RAYN_MULADD_FUSED", "0") == "1"
LEGACY = os.environ.get("RAYN_B200_LEGACY", "0") == "1"
LIB_NAME = "librayn_b200_fma.so" if MULADD_FUSED else ("librayn_b200_legacy.so" if LEGACY else "librayn_b200.so")
LIB_NAME = os.environ.get("RAYN_B200_LIB", LIB_NAME)  # tuning experiments: an explicitly named build
LIB_PATH = os.path.join(_HERE, "_build", LIB_NAME)
HOSTLIB_PATH = os.path.join(_HERE, "_build", "librayn_hostinputs.so")

RAYN_MAX_HITABLES = 1024
RAYN_MAX_MATERIALS = 1024
RAYN_MAX_LIGHTS = 256
RAYN_MAX_SDF_HITABLES = 16
RAYN_FIS_TABLE_SIZE = 512

RAYN_OK = 0
RAYN_ERR_INVALID_ARG = 1
RAYN_ERR_UNSUPPORTED = 2
RAYN_ERR_CUDA = 3
RAYN_ERR_OOM = 4
RAYN_ERR_NO_SCENE = 5
RAYN_ERR_NO_DEVICE = 6
RAYN_ERR_NCCL = 7
COMM_ID_BYTES = 128

HITABLE_SPHERE, HITABLE_MANDELBOX, HITABLE_MANDELBULB = 0, 1, 2
MATERIAL_LAMBERTIAN, MATERIAL_DIELECTRIC, MATERIAL_SKY, MATERIAL_EMISSIVE = 0, 1, 2, 3
CAMERA_PINHOLE, CAMERA_THINLENS, CAMERA_ORTHOGRAPHIC = 0, 1, 2
MEM_HOST, MEM_DEVICE = 0, 1
POST_COLOR_PLUS_BACKGROUND, POST_COLOR_ALPHA, POST_COLOR_ONLY, POST_BACKGROUND, POST_WORLD_NORMAL, POST_ALPHA = range(6)
POST_BYTES = (3, 4, 3, 3, 3, 1)
FLAG_TIMING, FLAG_SIMPLE_MARCH, FLAG_NO_GRAPH, FLAG_NO_DIV3, FLAG_NO_FOLD_ALL = 1, 2, 16, 32, 64
FLAG_SCENE_TABLES = 4
STAT_KERNELS = 12
KERNEL_NAMES = ["raygen", "extend", "bin", "shade_pre", "shadow", "shade_post", "compact", "resolve", "misc", "normals", "extend_spheres", "gather"]

f32 = C.c_float
i32 = C.c_int32
i64 = C.c_int64
fp = C.POINTER(C.c_float)


class RaynHitable(C.Structure):
    _fields_ = [("kind", i32), ("material", i32), ("center", f32 * 3), ("radius", f32),
                ("iterations", i32), ("box_l", f32), ("min_rad_sq", f32), ("fixed_rad_sq", f32),
                ("scale", f32), ("bulb_power", i32), ("bulb_bailout", f32), ("center_velocity", f32 * 3)]


class RaynMaterial(C.Structure):
    _fields_ = [("kind", i32), ("albedo", f32 * 3), ("roughness", f32), ("sky_top", f32 * 3),
                ("sky_bottom", f32 * 3), ("emission", f32 * 3)]


class RaynLight(C.Structure):
    _fields_ = [("pos", f32 * 3), ("rad", f32), ("emission", f32 * 3)]


class RaynCamera(C.Structure):
    _fields_ = [("kind", i32), ("half_size", f32 * 2), ("full_size", f32 * 2), ("half_pixel_size", f32),
                ("origin", f32 * 3), ("at", f32 * 3), ("up", f32 * 3), ("focus", f32 * 3), ("aperture", f32),
                ("origin_velocity", f32 * 3), ("at_velocity", f32 * 3), ("up_velocity", f32 * 3), ("focus_velocity", f32 * 3),
                ("aperture_rate", f32)]


class RaynVolume(C.Structure):
    _fields_ = [("has_scattering", i32), ("coeff_scattering", f32), ("has_extinction", i32),
                ("coeff_extinction", f32)]


class RaynRenderConsts(C.Structure):
    _fields_ = [("world_radius", f32), ("sdf_detail_scale", f32), ("max_marches", i32),
                ("max_vis_marches", i32)]


class RaynSceneDesc(C.Structure):
    _fields_ = [("n_hitables", i32), ("hitables", C.POINTER(RaynHitable)), ("n_materials", i32),
                ("materials", C.POINTER(RaynMaterial)), ("n_lights", i32), ("lights", C.POINTER(RaynLight)),
                ("camera", RaynCamera), ("volume", RaynVolume), ("consts", RaynRenderConsts)]


class RaynFrameDesc(C.Structure):
    _fields_ = [("width", i32), ("height", i32), ("tile_w", i32), ("tile_h", i32), ("samples", i32),
                ("max_bounces", i32), ("volume_marches", i32), ("frame", i32), ("t0", f32), ("t1", f32),
                ("sets_1d", i32), ("sets_2d", i32), ("samples_1d", C.c_void_p), ("samples_2d", C.c_void_p),
                ("scramble", C.c_void_p), ("fis_inverse_cdf", C.c_void_p), ("input_space", i32),
                ("tile_offset", i32), ("tile_stride", i32), ("tile_list", C.POINTER(i32)), ("n_tile_list", i32)]


class RaynFilmPlanes(C.Structure):
    _fields_ = [("color", C.c_void_p), ("alpha", C.c_void_p), ("background", C.c_void_p),
                ("normal", C.c_void_p), ("space", i32)]


class RaynConfig(C.Structure):
    _fields_ = [("device", i32), ("max_paths_per_pass", i64), ("flags", i32)]


class RaynStats(C.Structure):
    _fields_ = [("launches", i64), ("passes", i64), ("paths", i64), ("extend_rays", i64),
                ("shade_lanes", i64), ("shadow_rays", i64), ("sdf_evals_extend", i64),
                ("sdf_evals_shadow", i64), ("kernel_ms", f32 * STAT_KERNELS),
                ("kernel_launches", i64 * STAT_KERNELS), ("total_ms", f32), ("sdf_evals_normals", i64),
                ("bulb_iters_extend", i64), ("bulb_iters_shadow", i64), ("reserved_", i64),
                ("march_trips_extend", i64), ("march_trips_shadow", i64)]


# name -> (restype, argtypes); this table is also what the CPU test checks the header against
SYMBOLS = {
    "rayn_b200_abi_version": (i32, []),
    "rayn_b200_muladd_fused": (i32, []),
    "rayn_b200_comm_unique_id": (i32, [C.c_void_p]),
    "rayn_b200_comm_init_rank": (i32, [C.c_void_p, C.c_void_p, i32, i32]),
    "rayn_b200_comm_init_all": (i32, [C.POINTER(C.c_void_p), i32]),
    "rayn_b200_comm_destroy": (i32, [C.c_void_p]),
    "rayn_b200_comm_info": (i32, [C.c_void_p, C.POINTER(i32), C.POINTER(i32)]),
    "rayn_b200_shard_tiles": (i32, [i32, i32, i32, i32, i32, i32, C.POINTER(i32), i32]),
    "rayn_b200_render_frame_sharded": (i32, [C.c_void_p, C.POINTER(RaynFrameDesc), C.POINTER(RaynFilmPlanes)]),
    "rayn_b200_render_frame_multi": (i32, [C.POINTER(C.c_void_p), i32, C.POINTER(RaynFrameDesc), C.POINTER(RaynFilmPlanes)]),
    "rayn_b200_film_gather": (i32, [C.c_void_p, i32, i32, i32, i32, C.POINTER(RaynFilmPlanes)]),
    "rayn_b200_sync": (i32, [C.c_void_p]),
    "rayn_b200_kat_sdf_dist2": (i32, [C.c_void_p, C.POINTER(RaynHitable), i32, i64, fp, fp]),
    "rayn_b200_kat_fastdiv": (i32, [C.c_void_p, f32, C.c_uint32, i64, C.POINTER(i64)]),
    "rayn_b200_create": (i32, [C.POINTER(RaynConfig), C.POINTER(C.c_void_p)]),
    "rayn_b200_destroy": (None, [C.c_void_p]),
    "rayn_b200_last_error": (C.c_char_p, [C.c_void_p]),
    "rayn_b200_upload_scene": (i32, [C.c_void_p, C.POINTER(RaynSceneDesc)]),
    "rayn_b200_render_frame": (i32, [C.c_void_p, C.POINTER(RaynFrameDesc), C.POINTER(RaynFilmPlanes)]),
    "rayn_b200_get_stats": (i32, [C.c_void_p, C.POINTER(RaynStats)]),
    "rayn_b200_film_slab_floats": (i64, [i32, i32, i32]),
    "rayn_b200_film_pack_tiles": (i32, [C.c_void_p, i32, i32, i32, i32, C.POINTER(i32), i32, C.POINTER(RaynFilmPlanes), C.c_void_p]),
    "rayn_b200_film_unpack_tiles": (i32, [C.c_void_p, i32, i32, i32, i32, C.POINTER(i32), i32, C.c_void_p, C.POINTER(RaynFilmPlanes)]),
    "rayn_b200_film_postprocess": (i32, [C.c_void_p, i32, i32, i32, C.POINTER(RaynFilmPlanes), C.c_void_p, i32]),
    "rayn_b200_host_rd_tables": (i32, [i32, i32, i32, C.c_uint64, fp, fp]),
    "rayn_b200_host_scramble": (i32, [i32, i32, fp]),
    "rayn_b200_host_fis_blackman_harris": (i32, [f32, fp]),
    "rayn_b200_device_frame_inputs": (i32, [C.c_void_p, i32, i32, i32, i32, i32, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p]),
    "rayn_b200_host_tile_grid": (i32, [i32, i32, i32, i32, C.POINTER(i32), C.POINTER(i32)]),
    "rayn_b200_kat_detmath": (i32, [C.c_void_p, i32, i64, fp, fp, fp]),
    "rayn_b200_kat_sdf_dist": (i32, [C.c_void_p, C.POINTER(RaynHitable), i64, fp, fp]),
    "rayn_b200_kat_sdf_hit": (i32, [C.c_void_p, C.POINTER(RaynHitable), C.POINTER(RaynRenderConsts), i64, fp, fp, fp, f32, i32, fp]),
    "rayn_b200_kat_occluded": (i32, [C.c_void_p, i64, fp, fp, fp]),
    "rayn_b200_kat_closest_hit": (i32, [C.c_void_p, i32, i64, fp, fp, fp, C.POINTER(i32)]),
    "rayn_b200_kat_light_sample": (i32, [C.c_void_p, C.POINTER(RaynLight), i64, fp, fp, fp, fp, fp]),
    "rayn_b200_kat_light_sample_volume": (i32, [C.c_void_p, C.POINTER(RaynLight), i64, fp, fp, fp, fp, fp, fp]),
    "rayn_b200_kat_bsdf": (i32, [C.c_void_p, C.POINTER(RaynMaterial), i64, fp, fp, fp, fp, fp, fp, fp, fp]),
    "rayn_b200_debug_sdf_variant": (i32, [C.c_void_p, i32]),
    "rayn_b200_debug_enable_queue_log": (i32, [C.c_void_p, i32]),
    "rayn_b200_debug_read_queue_log": (i64, [C.c_void_p, C.POINTER(i32), i64]),
}

HOST_SYMBOLS = ("rayn_b200_host_rd_tables", "rayn_b200_host_scramble", "rayn_b200_host_fis_blackman_harris", "rayn_b200_host_tile_grid")

_lib = None
_hostlib = None


class RaynError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"rayn_b200 error {code}: {msg}")
        self.code = code


def lib():
    """Load librayn_b200.so (built in-tree by rayn_b200.build).  Fails loudly if absent."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `python -m rayn_b200.build` "
                "(the render path is CUDA only; there is no fallback)")
        l = C.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(l, name)  # AttributeError if the .so lacks a declared symbol
            fn.restype = res
            fn.argtypes = args
        _lib = l
    return _lib


def host_lib():
    """The pure-CPU builders of the host-owned frame inputs (the rayn_b200_host_* entry points of the header), from
    librayn_hostinputs.so: the same object code as in librayn_b200.so, without mapping the CUDA library."""
    global _hostlib
    if _hostlib is None:
        if not os.path.exists(HOSTLIB_PATH):
            raise ImportError(f"{HOSTLIB_PATH} is missing: build it with `python -m rayn_b200.build`")
        l = C.CDLL(HOSTLIB_PATH)
        for name in HOST_SYMBOLS:
            fn = getattr(l, name)
            fn.restype, fn.argtypes = SYMBOLS[name]
        _hostlib = l
    return _hostlib


def check(code, ctx=None):
    if code != RAYN_OK:
        msg = lib().rayn_b200_last_error(ctx) if (_lib is not None or ctx is not None) else None
        raise RaynError(code, msg.decode() if msg else "?")
