"""ctypes binding of the C ABI declared in include/ftkb200.h (libftkb200.so, built in-tree).

This is the reference-side binding a Python caller would use; it has no torch dependency.
There is no fallback: if the shared library is missing, loading raises.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libftkb200.so")

ABI_VERSION = 2
OK, ERR_INVALID, ERR_NO_DEVICE, ERR_CUDA, ERR_NOMEM, ERR_OVERFLOW = range(6)
SOURCE_NONE, SOURCE_GIVEN, SOURCE_DERIVED = 0, 1, 2
MEM_HOST, MEM_DEVICE, MEM_DEVICE_BORROW = 0, 1, 2
COORDS_SIMPLE, COORDS_BOUNDS, COORDS_RECTILINEAR, COORDS_EXPLICIT = range(4)
SYN_MOVING_EXTREMUM, SYN_WOVEN, SYN_DOUBLE_GYRE, SYN_ABC, SYN_MERGER, SYN_TORNADO = range(6)


class Config(C.Structure):
    _fields_ = [
        ("abi_version", C.c_int32), ("nd", C.c_int32), ("dims", C.c_int32 * 3), ("lb", C.c_int32 * 3), ("ub", C.c_int32 * 3),
        ("scalar_source", C.c_int32), ("vector_source", C.c_int32), ("jacobian_source", C.c_int32),
        ("jacobian_symmetric", C.c_int32), ("robust_detection", C.c_int32), ("compute_degrees", C.c_int32),
        ("use_type_filter", C.c_int32), ("type_filter", C.c_uint32), ("start_timestep", C.c_int32), ("device", C.c_int32),
        ("resolution_init", C.c_double), ("point_capacity", C.c_uint64),
        ("slab_offset", C.c_int32), ("slab_global_dim", C.c_int32), ("slab_global_lb", C.c_int32), ("slab_global_ub", C.c_int32),
    ]


class IpcHandle(C.Structure):
    _fields_ = [("bytes", C.c_uint8 * 64), ("offset", C.c_uint64)]


class Stats(C.Structure):
    _fields_ = [
        ("simplices_tested", C.c_uint64), ("cells_scanned", C.c_uint64), ("cells_refined", C.c_uint64), ("points", C.c_uint64),
        ("kernel_launches", C.c_uint64), ("h2d_bytes", C.c_uint64), ("d2h_bytes", C.c_uint64),
        ("ms_derive", C.c_double), ("ms_scan", C.c_double), ("ms_test", C.c_double), ("ms_finalize_device", C.c_double),
        ("ms_finalize_host", C.c_double), ("last_ms_scan", C.c_double), ("last_ms_derive", C.c_double),
        ("scaling_factor", C.c_double), ("resolution", C.c_double),
        ("scan_launches", C.c_uint64), ("sweeps_repeated", C.c_uint64),
        ("ms_sort_wall", C.c_double), ("ms_trace_wall", C.c_double),
    ]

    def as_dict(self):
        return {name: getattr(self, name) for name, _ in self._fields_}


POINT_DTYPE = np.dtype([
    ("corner", np.int32, 4), ("simplex_type", np.int32), ("ordinal", np.int32), ("timestep", np.int32),
    ("cp_type", np.uint32), ("x", np.float64, 3), ("t", np.float64), ("scalar", np.float64),
], align=True)
assert POINT_DTYPE.itemsize == 72

# ftkb_curve_point / ftkb_curve_info (trajectory post-processing)
CURVE_POINT_DTYPE = np.dtype([("p", POINT_DTYPE), ("v", np.float64, 3), ("id", np.int32), ("reserved", np.int32)], align=True)
assert CURVE_POINT_DTYPE.itemsize == 104
CURVE_INFO_DTYPE = np.dtype([
    ("id", np.int32), ("loop", np.int32), ("complete", np.int32), ("consistent_type", np.uint32), ("first", np.uint64), ("count", np.uint64),
    ("tmin", np.float64), ("tmax", np.float64), ("bbmin", np.float64, 3), ("bbmax", np.float64, 3),
    ("smin", np.float64), ("smax", np.float64), ("persistence", np.float64), ("vmmin", np.float64), ("vmmax", np.float64),
], align=True)
assert CURVE_INFO_DTYPE.itemsize == 136

class Piece(C.Structure):
    """ftkb_piece: planes [first, first + count) of a snapshot's slowest axis, in device memory"""
    _fields_ = [("scalar", C.c_void_p), ("vector", C.c_void_p), ("jacobian", C.c_void_p), ("first", C.c_int32), ("count", C.c_int32),
                ("stream", C.c_void_p), ("has_stream", C.c_int32), ("reserved", C.c_int32)]


# every symbol include/ftkb200.h declares
EXPORTS = [
    "ftkb_abi_version", "ftkb_device_count", "ftkb_create", "ftkb_destroy", "ftkb_last_error", "ftkb_push_snapshot",
    "ftkb_push_synthetic", "ftkb_update_timestep", "ftkb_advance_timestep", "ftkb_finalize", "ftkb_current_timestep",
    "ftkb_last_layer_resolution", "ftkb_set_resolution", "ftkb_num_points", "ftkb_get_points", "ftkb_import_points",
    "ftkb_num_trajectories", "ftkb_get_trajectories", "ftkb_get_component_labels", "ftkb_get_degrees", "ftkb_get_last_worklist", "ftkb_get_stats",
    "ftkb_reset_stats", "ftkb_synchronize", "ftkb_timer_start", "ftkb_timer_stop", "ftkb_mesh_ntypes", "ftkb_mesh_unit_simplex", "ftkb_mesh_scope_type",
    "ftkb_mesh_sides", "ftkb_mesh_side_of",
    "ftkb_curveset_create", "ftkb_get_curveset", "ftkb_curveset_destroy", "ftkb_curveset_post_process", "ftkb_curveset_size",
    "ftkb_curveset_get", "ftkb_curveset_last_error", "ftkb_curveset_slice", "ftkb_get_live_curveset", "ftkb_group_get_live_curveset",
    "ftkb_ipc_export", "ftkb_ipc_import", "ftkb_ipc_close", "ftkb_export_layer_cells", "ftkb_push_snapshot_remote",
    "ftkb_set_streaming_trajectories", "ftkb_get_trajectory_complete", "ftkb_online_create", "ftkb_online_destroy", "ftkb_online_grow", "ftkb_online_grow_prepared",
    "ftkb_online_size", "ftkb_online_get", "ftkb_set_coords", "ftkb_set_producer_stream", "ftkb_get_layer",
    "ftkb_group_create", "ftkb_group_destroy", "ftkb_group_last_error", "ftkb_group_set_coords",
    "ftkb_group_set_streaming_trajectories", "ftkb_group_push_snapshot", "ftkb_group_push_synthetic",
    "ftkb_group_push_snapshot_device", "ftkb_group_set_producer_stream", "ftkb_group_push_pieces_device", "ftkb_group_get_slab",
    "ftkb_group_advance_timestep", "ftkb_group_update_timestep", "ftkb_group_finalize", "ftkb_group_get_stats",
    "ftkb_host_alloc", "ftkb_host_free", "ftkb_push_snapshot_f32", "ftkb_bind_thread_to_device",
]

_lib = None


class FTKBError(RuntimeError):
    def __init__(self, code, message):
        super().__init__(f"ftkb error {code}: {message}")
        self.code = code


def lib():
    """Load libftkb200.so (raises if it has not been built: python -m ftk_b200.build)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise FileNotFoundError(f"{LIB_PATH} is missing: build it with `python -m ftk_b200.build` (there is no fallback path)")
    L = C.CDLL(LIB_PATH)
    vp, u64p = C.c_void_p, C.POINTER(C.c_uint64)
    L.ftkb_create.argtypes = [C.POINTER(Config), C.POINTER(vp)]
    L.ftkb_destroy.argtypes = [vp]
    L.ftkb_destroy.restype = None
    L.ftkb_last_error.argtypes = [vp]
    L.ftkb_last_error.restype = C.c_char_p
    L.ftkb_push_snapshot.argtypes = [vp, vp, vp, vp, C.c_int]
    L.ftkb_push_synthetic.argtypes = [vp, C.c_int, C.POINTER(C.c_double), C.c_int, C.c_double]
    for name in ("ftkb_update_timestep", "ftkb_advance_timestep", "ftkb_finalize", "ftkb_reset_stats", "ftkb_synchronize", "ftkb_timer_start"):
        getattr(L, name).argtypes = [vp]
    L.ftkb_timer_stop.argtypes = [vp, C.POINTER(C.c_double)]
    L.ftkb_current_timestep.argtypes = [vp, C.POINTER(C.c_int32)]
    L.ftkb_last_layer_resolution.argtypes = [vp, C.POINTER(C.c_double)]
    L.ftkb_set_resolution.argtypes = [vp, C.c_double]
    L.ftkb_num_points.argtypes = [vp, u64p]
    L.ftkb_get_points.argtypes = [vp, vp, C.c_uint64]
    L.ftkb_import_points.argtypes = [vp, vp, C.c_uint64]
    L.ftkb_num_trajectories.argtypes = [vp, u64p]
    L.ftkb_get_trajectories.argtypes = [vp, vp, vp, vp]
    L.ftkb_get_component_labels.argtypes = [vp, vp]
    L.ftkb_get_degrees.argtypes = [vp, vp]
    L.ftkb_get_last_worklist.argtypes = [vp, vp, C.c_uint64, u64p]
    L.ftkb_get_stats.argtypes = [vp, C.POINTER(Stats)]
    L.ftkb_mesh_ntypes.argtypes = [C.c_int, C.c_int, C.c_int]
    L.ftkb_mesh_unit_simplex.argtypes = [C.c_int, C.c_int, C.c_int, vp]
    L.ftkb_mesh_scope_type.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int]
    L.ftkb_mesh_sides.argtypes = [C.c_int, C.c_int, C.c_int, vp]
    L.ftkb_mesh_side_of.argtypes = [C.c_int, C.c_int, C.c_int, vp]
    L.ftkb_curveset_create.argtypes = [vp, C.c_uint64, vp, vp, vp, C.c_uint64, C.POINTER(vp)]
    L.ftkb_get_curveset.argtypes = [vp, C.POINTER(vp)]
    L.ftkb_get_live_curveset.argtypes = [vp, C.POINTER(C.c_int32), C.POINTER(vp)]
    L.ftkb_group_get_live_curveset.argtypes = [vp, C.POINTER(C.c_int32), C.POINTER(vp)]
    L.ftkb_curveset_destroy.argtypes = [vp]
    L.ftkb_curveset_destroy.restype = None
    L.ftkb_curveset_post_process.argtypes = [vp, C.c_char_p]
    L.ftkb_curveset_size.argtypes = [vp, u64p, u64p]
    L.ftkb_curveset_get.argtypes = [vp, vp, vp]
    L.ftkb_curveset_slice.argtypes = [vp, C.c_int32, vp, C.c_uint64, u64p]
    L.ftkb_ipc_export.argtypes = [vp, C.POINTER(IpcHandle)]
    L.ftkb_ipc_import.argtypes = [C.POINTER(IpcHandle), C.c_int, C.POINTER(vp)]
    L.ftkb_ipc_close.argtypes = [vp, C.POINTER(IpcHandle)]
    L.ftkb_export_layer_cells.argtypes = [vp, C.c_int, C.POINTER(vp), u64p, C.POINTER(C.c_double)]
    L.ftkb_push_snapshot_remote.argtypes = [vp, vp, vp, vp, C.c_double]
    L.ftkb_curveset_last_error.argtypes = [vp]
    L.ftkb_set_streaming_trajectories.argtypes = [vp, C.c_int]
    L.ftkb_set_coords.argtypes = [vp, C.c_int, vp, C.c_uint64]
    L.ftkb_set_producer_stream.argtypes = [vp, vp, C.c_int]
    L.ftkb_get_layer.argtypes = [vp, C.c_int, vp, vp]
    L.ftkb_group_create.argtypes = [C.POINTER(Config), C.POINTER(C.c_int32), C.c_int32, C.c_int32, C.POINTER(vp)]
    L.ftkb_group_destroy.argtypes = [vp]
    L.ftkb_group_destroy.restype = None
    L.ftkb_group_last_error.argtypes = [vp]
    L.ftkb_group_last_error.restype = C.c_char_p
    L.ftkb_group_set_coords.argtypes = [vp, C.c_int, vp, C.c_uint64]
    L.ftkb_group_set_streaming_trajectories.argtypes = [vp, C.c_int]
    L.ftkb_group_push_snapshot.argtypes = [vp, vp, vp, vp]
    L.ftkb_group_push_snapshot_device.argtypes = [vp, vp, vp, vp]
    L.ftkb_group_set_producer_stream.argtypes = [vp, vp, C.c_int]
    L.ftkb_group_push_pieces_device.argtypes = [vp, C.POINTER(Piece), C.c_int32]
    L.ftkb_group_get_slab.argtypes = [vp, C.c_int32, C.POINTER(C.c_int32)]
    L.ftkb_group_push_synthetic.argtypes = [vp, C.c_int, C.POINTER(C.c_double), C.c_int, C.c_double]
    L.ftkb_group_advance_timestep.argtypes = [vp]
    L.ftkb_group_update_timestep.argtypes = [vp]
    L.ftkb_group_finalize.argtypes = [vp, C.POINTER(vp)]
    L.ftkb_group_get_stats.argtypes = [vp, C.POINTER(Stats), C.POINTER(C.c_int32)]
    L.ftkb_host_alloc.argtypes = [C.c_uint64, C.POINTER(vp)]
    L.ftkb_host_free.argtypes = [vp]
    L.ftkb_push_snapshot_f32.argtypes = [vp, vp, vp]
    L.ftkb_bind_thread_to_device.argtypes = [C.c_int]
    L.ftkb_host_free.restype = None
    L.ftkb_get_trajectory_complete.argtypes = [vp, vp]
    L.ftkb_online_create.argtypes = [C.c_int, vp, vp, C.POINTER(vp)]
    L.ftkb_online_destroy.argtypes = [vp]
    L.ftkb_online_destroy.restype = None
    L.ftkb_online_grow.argtypes = [vp, vp, C.c_uint64]
    L.ftkb_online_grow_prepared.argtypes = [vp, vp, C.c_uint64]
    L.ftkb_online_size.argtypes = [vp, u64p, u64p]
    L.ftkb_online_get.argtypes = [vp, vp, vp, vp, vp]
    L.ftkb_curveset_last_error.restype = C.c_char_p
    _lib = L
    return L


def ipc_export(dev_ptr):
    """bytes of an ftkb_ipc_handle for a device pointer of this process (send it to a peer process of the same node)"""
    h = IpcHandle()
    rc = lib().ftkb_ipc_export(C.c_void_p(int(dev_ptr)), C.byref(h))
    if rc:
        raise FTKBError(rc, "ipc_export failed (memory not allocated with cudaMalloc?)")
    return bytes(h)


def ipc_import(handle_bytes, device):
    """map a peer process's allocation; returns the device pointer (int) valid in this process"""
    h = IpcHandle.from_buffer_copy(handle_bytes)
    out = C.c_void_p()
    rc = lib().ftkb_ipc_import(C.byref(h), int(device), C.byref(out))
    if rc:
        raise FTKBError(rc, "ipc_import failed")
    return int(out.value)


def ipc_close(dev_ptr, handle_bytes):
    """unmap a peer allocation mapped with ipc_import"""
    h = IpcHandle.from_buffer_copy(handle_bytes)
    rc = lib().ftkb_ipc_close(C.c_void_p(int(dev_ptr)), C.byref(h))
    if rc:
        raise FTKBError(rc, "ipc_close failed")
