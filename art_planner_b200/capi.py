"""ctypes binding of libartp.so -- the C ABI declared in include/artp.h.

The product path fails loudly when the CUDA library is missing or unusable: there is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libartp.so")

ARTP_OK, ARTP_E_INVALID, ARTP_E_NOMAP, ARTP_E_CUDA, ARTP_E_LIMIT, ARTP_E_NOWEIGHTS, ARTP_E_WINDOW = 0, -1, -2, -3, -4, -5, -6


class ArtpError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"artp error {code}: {msg}")
        self.code = code


class ArtpParams(C.Structure):
    _fields_ = [(n, C.c_double) for n in (
        "torso_length", "torso_width", "torso_height", "torso_off_x", "torso_off_y", "torso_off_z",
        "feet_off_x", "feet_off_y", "feet_off_z", "reach_x", "reach_y", "reach_z")] + [
        ("unknown_space_untraversable", C.c_int), ("use_directional_cost", C.c_int),
        ("max_lon_vel", C.c_double), ("max_lat_vel", C.c_double), ("max_ang_vel", C.c_double),
        ("cost_w_energy", C.c_float), ("cost_w_time", C.c_float), ("cost_w_risk", C.c_float),
        ("risk_threshold", C.c_float), ("device", C.c_int)]


class ArtpSamplerParams(C.Structure):
    _fields_ = [("max_roll_pert", C.c_double), ("max_pitch_pert", C.c_double), ("sample_from_distribution", C.c_int),
                ("low", C.c_double * 2), ("high", C.c_double * 2)]


class ArtpSe3Space(C.Structure):
    _fields_ = [("low", C.c_double * 3), ("high", C.c_double * 3), ("longest_valid_segment_fraction", C.c_double)]


class ArtpBasicParams(C.Structure):
    _fields_ = [("traversability_thres", C.c_float), ("unknown_space_untraversable", C.c_int)] + [(n, C.c_double) for n in (
        "foothold_margin", "foothold_margin_max_hole_size", "foothold_margin_max_drop", "foothold_margin_max_drop_search_radius",
        "foothold_margin_min_step", "foothold_size")]


class ArtpGrid(C.Structure):
    _fields_ = [("elevation", C.c_void_p), ("traversability_thresholded", C.c_void_p), ("rows", C.c_int), ("cols", C.c_int),
                ("res", C.c_double), ("cx", C.c_double), ("cy", C.c_double)]


class ArtpStats(C.Structure):
    _fields_ = [("poses_checked", C.c_uint64), ("poses_deferred", C.c_uint64), ("kernel_launches", C.c_uint64),
                ("last_deferred", C.c_uint32), ("last_launches", C.c_uint32), ("last_queued_boxes", C.c_uint32),
                ("last_queued_warp_stage", C.c_uint32), ("last_queued_reach_stage", C.c_uint32),
                ("last_reach_plane_stage", C.c_uint32)]


_lib = None


def load():
    """Load libartp.so (raises if it is missing: build it with art_planner_b200.build.build())."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise FileNotFoundError(f"{LIB_PATH} not built; run `python -m art_planner_b200.build` (needs nvcc)")
    lib = C.CDLL(LIB_PATH)
    vp, sz, i32, dbl = C.c_void_p, C.c_size_t, C.c_int, C.c_double
    lib.artp_create.argtypes = [C.POINTER(ArtpParams), C.POINTER(vp)]
    lib.artp_destroy.argtypes = [vp]
    lib.artp_destroy.restype = None
    lib.artp_last_error.argtypes = [vp]
    lib.artp_last_error.restype = C.c_char_p
    lib.artp_set_map.argtypes = [vp, vp, vp, i32, i32, dbl, dbl, dbl]
    lib.artp_has_map.argtypes = [vp]
    lib.artp_check_poses.argtypes = [vp, vp, sz, vp]
    lib.artp_check_poses_device.argtypes = [vp, vp, sz, vp, vp]
    lib.artp_check_poses_f32.argtypes = [vp, vp, sz, vp]
    lib.artp_check_poses_f32_device.argtypes = [vp, vp, sz, vp, vp]
    lib.artp_check_motions.argtypes = [vp, vp, vp, sz, i32, vp]
    lib.artp_check_motions_device.argtypes = [vp, vp, vp, sz, i32, vp, vp]
    lib.artp_valid_segment_count.argtypes = [C.POINTER(ArtpSe3Space), vp, vp, sz, vp]
    lib.artp_check_motions_segments.argtypes = [vp, vp, vp, sz, vp, C.POINTER(ArtpSe3Space), vp, vp]
    lib.artp_edge_matrix_from_states.argtypes = [vp, vp, sz, vp]
    lib.artp_motion_cost_states.argtypes = [vp, vp, vp, sz, vp, vp, vp]
    lib.artp_check_edge_interiors.argtypes = [vp, vp, vp, sz, vp, C.c_double, vp]
    lib.artp_check_edge_interiors_device.argtypes = [vp, vp, vp, sz, vp, sz, vp, vp, vp]
    u64 = C.c_uint64
    lib.artp_set_sampler.argtypes = [vp, C.POINTER(ArtpSamplerParams), vp, vp, vp, vp, vp, vp]
    lib.artp_estimate_normals.argtypes = [vp, C.c_double, vp, vp, vp, vp]
    lib.artp_compute_sample_cdf.argtypes = [vp, vp, vp, vp]
    lib.artp_sampler_uniforms.argtypes = [vp, u64, u64, sz, vp]
    lib.artp_sample_states.argtypes = [vp, vp, u64, u64, sz, vp, vp]
    lib.artp_sample_states_device.argtypes = [vp, vp, u64, u64, sz, vp, vp, vp]
    lib.artp_sample_valid.argtypes = [vp, u64, u64, sz, vp, sz, C.POINTER(C.c_size_t)]
    lib.artp_sample_valid_device.argtypes = [vp, u64, u64, sz, vp, sz, vp, vp]
    lib.artp_path_length_cost.argtypes = [vp, vp, vp, sz, vp]
    lib.artp_path_length_cost_device.argtypes = [vp, vp, vp, sz, vp, vp]
    lib.artp_compact_valid_device.argtypes = [vp, vp, sz, C.c_int64, vp, vp, vp]
    lib.artp_pack_valid_bits_device.argtypes = [vp, vp, sz, vp, vp]
    lib.artp_check_poses_bits_device.argtypes = [vp, vp, sz, vp, vp, vp]
    lib.artp_compact_valid_u32_device.argtypes = [vp, vp, sz, C.c_uint32, vp, vp, vp]
    lib.artp_set_map_window.argtypes = [vp, vp, vp, i32, i32, dbl, dbl, dbl, i32, i32]
    lib.artp_compact_bits_device.argtypes = [vp, vp, sz, C.c_int64, vp, vp, vp]
    lib.artp_get_stats.argtypes = [vp, C.POINTER(ArtpStats)]
    lib.artp_set_mode.argtypes = [vp, i32]
    lib.artp_poll_error.argtypes = [vp]
    lib.artp_process_basic.argtypes = [vp, vp, vp, vp, i32, i32, dbl, C.POINTER(ArtpBasicParams), vp, vp]
    lib.artp_debug_circular_kernel.argtypes = [i32, vp]
    lib.artp_host_alloc.restype = C.c_void_p
    lib.artp_host_alloc.argtypes = [sz]
    lib.artp_host_free.argtypes = [vp]
    lib.artp_debug_set_group_capacity.argtypes = [vp, i32]
    lib.artp_set_timing.argtypes = [vp, i32]
    lib.artp_get_last_timing.argtypes = [vp, C.POINTER(C.c_float)]
    lib.artp_get_last_stage_timing.argtypes = [vp, C.POINTER(C.c_float)]
    lib.artp_compute_change.argtypes = [vp, C.POINTER(ArtpGrid), C.POINTER(ArtpGrid), C.c_float, vp]
    lib.artp_compute_change_device.argtypes = [vp, C.POINTER(ArtpGrid), C.POINTER(ArtpGrid), C.c_float, vp, vp]
    lib.artp_roadmap_updates.argtypes = [vp, vp, sz, vp, sz, vp, vp]
    lib.artp_roadmap_updates_device.argtypes = [vp, vp, sz, vp, sz, vp, vp, vp]
    lib.artp_version.restype = C.c_char_p
    lib.artp_cost_weights_size.restype = C.c_size_t
    lib.artp_set_cost_weights.argtypes = [vp, vp, sz]
    lib.artp_update_features.argtypes = [vp]
    lib.artp_motion_cost.argtypes = [vp, vp, sz, vp]
    lib.artp_motion_cost_device.argtypes = [vp, vp, sz, vp, vp]
    lib.artp_combine_cost.argtypes = [vp, vp, sz, vp, vp]
    lib.artp_get_features.argtypes = [vp, vp, sz, C.POINTER(i32), C.POINTER(i32)]
    lib.artp_set_cnn_mode.argtypes = [vp, i32]
    lib.artp_get_cnn_timing.argtypes = [vp, C.POINTER(C.c_float)]
    _lib = lib
    return lib


def make_params(rp, device: int = 0, cost_weights=(0.0, 1.0, 5.0), risk_threshold=0.5) -> ArtpParams:
    p = ArtpParams()
    for name in ("torso_length", "torso_width", "torso_height", "torso_off_x", "torso_off_y", "torso_off_z",
                 "feet_off_x", "feet_off_y", "feet_off_z", "reach_x", "reach_y", "reach_z",
                 "max_lon_vel", "max_lat_vel", "max_ang_vel"):
        setattr(p, name, float(getattr(rp, name)))
    p.unknown_space_untraversable = int(rp.unknown_space_untraversable)
    p.use_directional_cost = int(rp.use_directional_cost)
    p.cost_w_energy, p.cost_w_time, p.cost_w_risk = [float(x) for x in cost_weights]
    p.risk_threshold = float(risk_threshold)
    p.device = int(device)
    return p


class HostBuffer:
    """A pinned host array from artp_host_alloc (cudaHostAlloc'd: reaches the device at PCIe line rate), as numpy."""

    def __init__(self, shape, dtype):
        import numpy as np
        self.lib = load()
        self.nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
        self.ptr = self.lib.artp_host_alloc(self.nbytes)
        if not self.ptr:
            raise ArtpError(ARTP_E_CUDA, "artp_host_alloc failed")
        buf = (C.c_char * self.nbytes).from_address(self.ptr)
        self.array = np.frombuffer(buf, dtype=dtype).reshape(shape)

    def close(self):
        if getattr(self, "ptr", None):
            self.array = None
            self.lib.artp_host_free(C.c_void_p(self.ptr))
            self.ptr = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
