"""ctypes binding of libtds_b200.so (the C ABI declared in include/tds_b200.h).

There is NO fallback: if the library is missing or a call fails, an exception is raised.  PyTorch is
used only as the owner of device memory and streams; raw device pointers cross the ABI.
"""
import ctypes
import os
from ctypes import POINTER, c_char_p, c_float, c_int32, c_int64, c_uint8, c_void_p

import torch

from . import _build

MAX_CLASSES = 32
MAX_AGENT_TYPES = 8
MAX_TL_STATES = 8
MAX_MAPS = 8

MODEL_BICYCLE = 0
MODEL_BICYCLE_NO_REVERSING = 1
MODEL_UNICYCLE = 2
MODEL_SIMPLE = 3
MODEL_ORIENTED = 4
METRIC_DISCS = 0
METRIC_IOU = 1
IMAGE_F32 = 0
IMAGE_U8 = 1
IMAGE_RANK = 2


class TdsError(RuntimeError):
    pass


class KinematicParams(ctypes.Structure):
    _fields_ = [("dt", c_float), ("max_acceleration", c_float), ("max_steering", c_float),
                ("max_yaw_rate", c_float), ("left_handed", c_int32), ("max_dx", c_float), ("max_dpsi", c_float),
                ("max_dv", c_float)]


class Palette(ctypes.Structure):
    _fields_ = [("n_classes", c_int32), ("active", c_uint8 * MAX_CLASSES), ("rank", c_uint8 * MAX_CLASSES), ("rgb", (c_uint8 * 3) * MAX_CLASSES),
                ("agent_type_class", c_int32 * MAX_AGENT_TYPES), ("direction_class", c_int32),
                ("tl_state_class", c_int32 * MAX_TL_STATES)]


class MapInfo(ctypes.Structure):
    _fields_ = [("n_verts", c_int32), ("n_faces", c_int32), ("raster_gx", c_int32), ("raster_gy", c_int32),
                ("raster_records", c_int32), ("offroad_gx", c_int32), ("offroad_gy", c_int32),
                ("offroad_entries", c_int32), ("raster_cell", c_float), ("offroad_cell", c_float),
                ("min_x", c_float), ("min_y", c_float), ("max_x", c_float), ("max_y", c_float),
                ("device_bytes", c_int64), ("raster_strips", c_int32), ("reserved", c_int32)]


# name -> (restype, argtypes); every symbol include/tds_b200.h declares
SIGNATURES = {
    "tds_version": (c_int32, []),
    "tds_last_error": (c_char_p, []),
    "tds_kinematic_step_fwd": (c_int32, [c_void_p, c_void_p, c_int32, c_void_p, c_void_p, c_int32, c_int64,
                                         POINTER(KinematicParams), c_void_p, c_void_p]),
    "tds_kinematic_step_bwd": (c_int32, [c_void_p, c_void_p, c_int32, c_void_p, c_void_p, c_int32, c_int64,
                                         POINTER(KinematicParams), c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "tds_collision_pairwise_fwd": (c_int32, [c_void_p, c_void_p, c_int64, c_int32, c_void_p, c_void_p]),
    "tds_collision_pairwise_bwd": (c_int32, [c_void_p, c_void_p, c_int64, c_int32, c_void_p, c_void_p, c_void_p, c_void_p]),
    "tds_collision_allpairs_fwd": (c_int32, [c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_int32, c_int32, c_int32,
                                             c_void_p, c_void_p, c_void_p]),
    "tds_collision_allpairs_bwd": (c_int32, [c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_int32, c_int32, c_int32,
                                             c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "tds_traffic_light_violation": (c_int32, [c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_int32, c_int32,
                                              c_float, c_void_p, c_void_p]),
    "tds_npc_advance": (c_int32, [c_void_p, c_void_p, c_int32, c_int32, c_void_p, c_int32, c_void_p, c_void_p, c_int32, c_int32,
                                  c_void_p, c_void_p, c_int32, c_int32, c_void_p]),
    "tds_waypoint_step": (c_int32, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int32, c_int32, c_float, c_void_p]),
    "tds_waypoint_gather": (c_int32, [c_void_p, c_void_p, c_void_p, c_int64, c_int32, c_int32, c_int32, c_void_p, c_void_p, c_void_p]),
    "tds_infraction_metrics": (c_int32, [c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p]),
    "tds_agent_boxes": (c_int32, [c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p]),
    "tds_rollout_loss": (c_int32, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p]),
    "tds_rollout_grad": (c_int32, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_float, c_float, c_float,
                                   c_int64, c_void_p, c_void_p]),
    "tds_agents_relative": (c_int32, [c_void_p, c_int32, c_int32, c_int32, c_int32, c_int32, c_void_p, c_void_p]),
    "tds_agents_relative_bwd": (c_int32, [c_void_p, c_void_p, c_int32, c_int32, c_int32, c_int32, c_int32, c_void_p, c_void_p]),
    "tds_nearest_agents_relative": (c_int32, [c_void_p, c_int32, c_int32, c_int32, c_int32, c_int32, c_float, c_void_p,
                                              c_void_p, c_void_p]),
    "tds_nearest_agents_relative_bwd": (c_int32, [c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_int32, c_int32, c_int32,
                                                  c_void_p, c_void_p]),
    "tds_sensing_noise": (c_int32, [c_void_p, c_void_p, c_int32, c_int32, c_int32, c_void_p, c_void_p]),
    "tds_sensing_occlusion": (c_int32, [c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_int32, c_void_p, c_void_p]),
    "tds_map_create": (c_void_p, [c_void_p, c_int32, c_void_p, c_int32, c_void_p, c_float, c_float]),
    "tds_map_destroy": (None, [c_void_p]),
    "tds_map_info": (c_int32, [c_void_p, POINTER(MapInfo)]),
    "tds_map_offroad_bound": (c_int32, [c_void_p, c_void_p, c_void_p, c_void_p]),
    "tds_map_segments": (c_int32, [c_void_p, c_void_p, c_void_p, c_void_p]),
    "tds_nearest_map_segments": (c_int32, [POINTER(c_void_p), c_int32, c_void_p, c_void_p, c_int32, c_int32, c_int32, c_float,
                                           c_void_p, c_void_p, c_void_p, c_void_p]),
    "tds_nearest_map_segments_bwd": (c_int32, [POINTER(c_void_p), c_int32, c_void_p, c_void_p, c_void_p, c_void_p, c_int32,
                                               c_int32, c_int32, c_void_p, c_void_p]),
    "tds_range_scan": (c_int32, [POINTER(c_void_p), c_int32, c_void_p, c_void_p, c_int32, c_int32, c_int32, c_int32, c_float,
                                 c_void_p, c_void_p, c_void_p, c_void_p]),
    "tds_range_scan_bwd": (c_int32, [POINTER(c_void_p), c_int32, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int32,
                                     c_int32, c_int32, c_int32, c_void_p, c_void_p]),
    "tds_time_to_collision": (c_int32, [c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_int32, c_float, c_void_p,
                                        c_void_p, c_void_p]),
    "tds_time_to_collision_bwd": (c_int32, [c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_int32, c_float, c_void_p,
                                            c_void_p, c_void_p, c_void_p, c_void_p]),
    "tds_offroad_fwd": (c_int32, [POINTER(c_void_p), c_int32, c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_int32,
                                  c_float, c_void_p, c_void_p, c_void_p]),
    "tds_offroad_bwd": (c_int32, [POINTER(c_void_p), c_int32, c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_int32,
                                  c_float, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "tds_raster_workspace_bytes": (c_int64, [c_int32, c_int32, c_int32, c_int32]),
    "tds_raster_set_timing_events": (None, [c_void_p, c_void_p]),
    "tds_raster_birdview_fmt": (c_int32, [POINTER(c_void_p), c_int32, c_void_p, c_int32, c_int32, c_int32,
                                          c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int32,
                                          c_void_p, c_void_p, c_int32, c_void_p, c_void_p, c_int32,
                                          c_void_p, c_void_p, c_int32,
                                          POINTER(Palette), c_float, c_int32, c_void_p, c_int32, c_void_p, c_void_p, c_void_p]),
    "tds_raster_rank_table": (c_int32, [POINTER(Palette), c_void_p, c_void_p]),
    "tds_raster_birdview": (c_int32, [POINTER(c_void_p), c_int32, c_void_p, c_int32, c_int32, c_int32,
                                      c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int32,
                                      c_void_p, c_void_p, c_int32, c_void_p, c_void_p, c_int32,
                                      c_void_p, c_void_p, c_int32,
                                      POINTER(Palette), c_float, c_int32, c_void_p, c_void_p, c_void_p]),
}

_LIB = None


def library_path() -> str:
    # TDS_B200_LIB selects an experimental build of the same ABI (profiling aid); default: the in-tree build
    return os.environ.get("TDS_B200_LIB") or _build.LIB_PATH


def load(build_if_missing: bool = True) -> ctypes.CDLL:
    """Loads libtds_b200.so; raises if it cannot be found/built (no CPU fallback exists)."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = library_path()
    if not os.path.exists(path):
        if not build_if_missing:
            raise TdsError(f"{path} is missing: run `python -m torchdrivesim_b200._build` (needs nvcc)")
        _build.build_library()
    lib = ctypes.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the ABI is incomplete
        fn.restype = res
        fn.argtypes = args
    _LIB = lib
    return lib


def check(code: int) -> None:
    if code != 0:
        raise TdsError(f"libtds_b200 error {code}: {load().tds_last_error().decode()}")


def ptr(t) -> int:
    """Device pointer of a contiguous CUDA tensor (None -> NULL)."""
    if t is None:
        return None
    if not t.is_cuda:
        raise TdsError("torchdrivesim_b200 ops need CUDA tensors: there is no CPU implementation")
    if not t.is_contiguous():
        raise TdsError("internal error: non-contiguous tensor passed to the C ABI")
    return t.data_ptr()


def stream_ptr(device=None) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def as_f32(t: torch.Tensor) -> torch.Tensor:
    return t.detach().to(torch.float32).contiguous()


def as_u8(t: torch.Tensor) -> torch.Tensor:
    t = t.detach()
    if t.dtype == torch.bool:
        return t.contiguous().view(torch.uint8)
    return (t != 0).contiguous().view(torch.uint8)


def as_i32(t: torch.Tensor) -> torch.Tensor:
    return t.detach().to(torch.int32).contiguous()
