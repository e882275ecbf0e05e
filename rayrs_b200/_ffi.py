"""ctypes bindings of include/rayrs_b200.h (CUDA backend) and of the C++ host mirror.

There is no fallback: if the native libraries are missing, importing anything that needs them
raises with the build command to run.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

_PKG = Path(__file__).resolve().parent
CUDA_LIB_PATH = _PKG / "librayrs_b200.so"
HOST_LIB_PATH = _PKG / "librayrs_host.so"

RRS_ABI_VERSION = 2
RRS_OK = 0
RRS_ERR_INVALID, RRS_ERR_NO_DEVICE, RRS_ERR_CUDA, RRS_ERR_TOO_DEEP, RRS_ERR_NOMEM, RRS_ERR_COMM = -1, -2, -3, -4, -5, -6
RRS_REF_LEAF = 0x80000000
RRS_REF_EMPTY = 0xFFFFFFFF
RRS_FLAG_COUNT_TRAVERSAL = 1
RRS_FLAG_TIME_PHASES = 2
RRS_FLAG_SPLIT_KERNELS = 4
RRS_FLAG_FORCE_QUEUES = 8
RRS_FLAG_FORCE_PATHLOOP = 16
RRS_FLAG_NO_L2_WINDOW = 32
RRS_FLAG_ENV_SAMPLING = 64
RRS_SCENE_NO_BRUTE, RRS_SCENE_NO_BRUTE_BOX, RRS_SCENE_NO_L2_PERSIST = 1, 2, 4


class RrsPrim(C.Structure):
    _fields_ = [("type", C.c_uint32), ("obj_id", C.c_uint32), ("material", C.c_uint32), ("emission", C.c_int32),
                ("v", C.c_double * 9)]


class RrsMaterial(C.Structure):
    _fields_ = [("tag", C.c_uint32), ("fresnel_kind", C.c_uint32), ("color", C.c_double * 3),
                ("spec_color", C.c_double * 3), ("alpha", C.c_double), ("ior", C.c_double)]


class RrsEmission(C.Structure):
    _fields_ = [("strength", C.c_double), ("color", C.c_double * 3)]


class RrsNode(C.Structure):
    _fields_ = [("lo0", C.c_float * 3), ("hi0", C.c_float * 3), ("lo1", C.c_float * 3), ("hi1", C.c_float * 3),
                ("ref0", C.c_uint32), ("ref1", C.c_uint32), ("flags", C.c_uint32), ("pad", C.c_uint32)]


class RrsNodeF64(C.Structure):
    _fields_ = [("lo0", C.c_double * 3), ("hi0", C.c_double * 3), ("lo1", C.c_double * 3), ("hi1", C.c_double * 3),
                ("ref0", C.c_uint32), ("ref1", C.c_uint32), ("flags", C.c_uint32), ("pad", C.c_uint32 * 5)]


class RrsSceneDesc(C.Structure):
    _fields_ = [("abi_version", C.c_uint32), ("n_prims", C.c_uint32), ("prims", C.POINTER(RrsPrim)),
                ("n_nodes", C.c_uint32), ("nodes", C.POINTER(RrsNode)), ("nodes_f64", C.POINTER(RrsNodeF64)),
                ("max_depth", C.c_uint32), ("n_materials", C.c_uint32), ("materials", C.POINTER(RrsMaterial)),
                ("n_emissions", C.c_uint32), ("emissions", C.POINTER(RrsEmission)),
                ("hdri_width", C.c_uint32), ("hdri_height", C.c_uint32), ("hdri_rgb", C.POINTER(C.c_float)),
                ("t_min", C.c_double), ("t_max", C.c_double), ("flags", C.c_uint32), ("refill_lanes", C.c_uint32)]


class RrsCamera(C.Structure):
    _fields_ = [("origin", C.c_double * 3), ("e_x", C.c_double * 3), ("e_y", C.c_double * 3),
                ("z_scaled", C.c_double * 3), ("width", C.c_double), ("height", C.c_double), ("ppc", C.c_uint32),
                ("x_pixels", C.c_uint32), ("y_pixels", C.c_uint32)]


class RrsRenderParams(C.Structure):
    _fields_ = [("width", C.c_uint32), ("height", C.c_uint32), ("spp", C.c_uint32), ("sample_offset", C.c_uint32),
                ("spp_total", C.c_uint32), ("max_bounces", C.c_uint32), ("seed", C.c_uint64),
                ("queue_capacity", C.c_uint32), ("flags", C.c_uint32)]


class RrsUniqueId(C.Structure):
    _fields_ = [("bytes", C.c_char * 128)]


class RrsBuildNode(C.Structure):
    _fields_ = [("box", C.c_double * 6), ("child", C.c_int32 * 2), ("first", C.c_uint32), ("count", C.c_uint32),
                ("kind", C.c_uint32), ("pad", C.c_uint32)]


class RrsRay(C.Structure):
    _fields_ = [("origin", C.c_double * 3), ("direction", C.c_double * 3)]


class RrsStats(C.Structure):
    _fields_ = [("rays", C.c_uint64), ("paths", C.c_uint64), ("kernel_launches", C.c_uint64),
                ("iterations", C.c_uint64), ("nan_pixels", C.c_uint64), ("negative_pixels", C.c_uint64),
                ("device_ms", C.c_double), ("extend_ms", C.c_double), ("shade_ms", C.c_double),
                ("generate_ms", C.c_double), ("nodes_visited", C.c_uint64), ("prims_tested", C.c_uint64),
                ("kernel_form", C.c_uint64), ("census_mismatch_pixels", C.c_uint64)]


RRS_FORM_WAVEFRONT, RRS_FORM_SPLIT, RRS_FORM_PATHLOOP = 0, 1, 2


# every symbol include/rayrs_b200.h declares: (name, restype, argtypes)
CUDA_SYMBOLS = {
    "rrs_scene_create": (C.c_int, [C.POINTER(RrsSceneDesc), C.c_int, C.POINTER(C.c_void_p)]),
    "rrs_scene_create_multi": (C.c_int, [C.POINTER(RrsSceneDesc), C.POINTER(C.c_int), C.c_int, C.POINTER(C.c_void_p)]),
    "rrs_scene_destroy": (None, [C.c_void_p]),
    "rrs_sample_range": (C.c_int, [C.c_uint32, C.c_uint32, C.c_uint32, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]),
    "rrs_comm_init_all": (C.c_int, [C.POINTER(C.c_int), C.c_int, C.POINTER(C.c_void_p)]),
    "rrs_comm_unique_id": (C.c_int, [C.POINTER(RrsUniqueId)]),
    "rrs_comm_init_rank": (C.c_int, [C.POINTER(RrsUniqueId), C.c_int, C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "rrs_comm_destroy": (None, [C.c_void_p]),
    "rrs_render_multi": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.c_void_p, C.POINTER(RrsCamera), C.POINTER(RrsRenderParams),
                                    C.c_void_p, C.c_int, C.POINTER(C.c_void_p)]),
    "rrs_render": (C.c_int, [C.c_void_p, C.POINTER(RrsCamera), C.POINTER(RrsRenderParams), C.c_void_p]),
    "rrs_render_accumulate": (C.c_int, [C.c_void_p, C.POINTER(RrsCamera), C.POINTER(RrsRenderParams), C.c_void_p, C.c_void_p]),
    "rrs_resolve": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.c_int, C.c_void_p]),
    "rrs_to_raw_bytes": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_double, C.c_void_p, C.c_int,
                                    C.c_void_p, C.c_void_p]),
    "rrs_intersect": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_int]),
    "rrs_material_evaluate": (C.c_int, [C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "rrs_material_evaluate_pdf": (C.c_int, [C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "rrs_background": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "rrs_env_sample": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "rrs_env_pdf": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "rrs_rng_uniforms": (C.c_int, [C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p]),
    "rrs_bvh_build": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_int, C.c_void_p, C.c_void_p,
                                 C.POINTER(C.c_uint32), C.POINTER(C.c_double)]),
    "rrs_stats": (C.c_int, [C.c_void_p, C.POINTER(RrsStats)]),
    "rrs_last_error": (C.c_char_p, []),
    "rrs_abi_version": (C.c_int, []),
    "rrs_device_count": (C.c_int, []),
}

HOST_SYMBOLS = {
    "rrh_last_error": (C.c_char_p, []),
    "rrh_scene_new": (C.c_void_p, [C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_int,
                                    C.c_uint32, C.c_void_p, C.c_uint64, C.c_uint64, C.c_double, C.c_double, C.c_int,
                                    C.c_int, C.c_int, C.c_uint32, C.c_uint32, C.c_int, C.POINTER(C.c_int), C.c_int, C.c_int, C.c_int]),
    "rrh_scene_free": (None, [C.c_void_p]),
    "rrh_scene_handle": (C.c_void_p, [C.c_void_p]),
    "rrh_scene_handle_at": (C.c_void_p, [C.c_void_p, C.c_uint32]),
    "rrh_scene_comm": (C.c_void_p, [C.c_void_p]),
    "rrh_scene_build_timing": (None, [C.c_void_p, C.POINTER(C.c_double)]),
    "rrh_scene_info": (None, [C.c_void_p, C.c_void_p, C.POINTER(C.c_double)]),
    "rrh_scene_copy": (None, [C.c_void_p] * 7),
    "rrh_camera_new": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_double, C.c_double, C.c_double, C.c_uint32,
                                  C.POINTER(RrsCamera)]),
    "rrh_load_mesh": (C.c_void_p, [C.c_char_p, C.c_int, C.POINTER(C.c_uint64)]),
    "rrh_load_obj_spheres": (C.c_void_p, [C.c_char_p, C.c_double, C.POINTER(C.c_uint64)]),
    "rrh_free": (None, [C.c_void_p]),
    "rrh_write_ply": (C.c_int, [C.c_char_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_int]),
    "rrh_ply_describe": (C.c_int, [C.c_char_p, C.c_uint64, C.c_char_p, C.c_uint64]),
}

_cuda = None
_host = None


def _load(path: Path, symbols: dict) -> C.CDLL:
    if not path.exists():
        raise ImportError(
            f"{path.name} is not built. rayrs_b200 has no CPU or Python fallback: run "
            "`python -m rayrs_b200.build` (needs nvcc) first.")
    lib = C.CDLL(str(path), mode=C.RTLD_GLOBAL)
    for name, (res, args) in symbols.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is missing: fail loudly
        fn.restype = res
        fn.argtypes = args
    return lib


def cuda_lib() -> C.CDLL:
    global _cuda
    if _cuda is None:
        _cuda = _load(CUDA_LIB_PATH, CUDA_SYMBOLS)
        if _cuda.rrs_abi_version() != RRS_ABI_VERSION:
            raise ImportError("librayrs_b200.so ABI version mismatch; rebuild")
    return _cuda


def host_lib() -> C.CDLL:
    global _host
    if _host is None:
        cuda_lib()
        _host = _load(HOST_LIB_PATH, HOST_SYMBOLS)
    return _host


class RayrsError(RuntimeError):
    """A non-zero status from the C ABI (the Rust shim would panic here)."""

    def __init__(self, status: int, message: str):
        super().__init__(f"rayrs_b200 status {status}: {message}")
        self.status = status


def check(status: int) -> None:
    if status != RRS_OK:
        raise RayrsError(status, cuda_lib().rrs_last_error().decode())
