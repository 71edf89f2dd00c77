"""ctypes binding of libb200_sixdof.so — the C ABI declared in include/b200_sixdof.h.

This is the only way the Python host reaches the integrator: there is no Python
or CPU implementation of the hot path in this package.  If the shared library
is missing or no CUDA device is visible, the calls below raise.
"""

from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libb200_sixdof.so")

ABI_VERSION = 3
MAX_EFFECTORS = 8

OK = 0
ERR_COMPONENT_NOT_FOUND = 1
ERR_VALUE_SIZE_MISMATCH = 2
ERR_INVALID_ARGUMENT = 3
ERR_UNSUPPORTED = 4
ERR_CUDA = 5
ERR_NO_DEVICE = 6
ERR_OUT_OF_MEMORY = 7

INTEGRATOR_RK4 = 0
INTEGRATOR_SEMI_IMPLICIT = 1
MATH_EXACT = 0
MATH_FAST = 1

EFF_GRAVITY_CONST = 1
EFF_DRAG_QUADRATIC = 2
EFF_THRUST_BODY = 3
EFF_WRENCH_BODY = 4
EFF_GRAVITY_FRAME = 5
EFF_GRAVITY_EDGES_NEWTON = 6
EFF_GRAVITY_EDGES_SOFTENED = 7
EFF_WRENCH_WORLD = 8
EFF_TORQUE_BODY_FOLD = 9
EFF_GRAVITY_J2 = 10
EFF_GRAVITY_EGM08 = 11
EFF_FLAG_WRENCH_LINEAR_FIRST = 1
TRAJ_FULL = 1

# every symbol include/b200_sixdof.h declares (tests/test_abi.py checks the export table against it)
SYMBOLS = [
    "b200_component_id", "b200_last_error", "b200_device_count", "b200_host_alloc", "b200_host_alloc_local", "b200_host_free",
    "b200_device_numa_node", "b200_host_node_of",
    "b200_sixdof_create", "b200_sixdof_destroy", "b200_sixdof_input_ids", "b200_sixdof_output_ids",
    "b200_sixdof_column_bytes", "b200_sixdof_upload", "b200_sixdof_download", "b200_sixdof_set_schedule",
    "b200_sixdof_clear_schedule", "b200_sixdof_step",
    "b200_sixdof_sync", "b200_sixdof_invoke_batch", "b200_sixdof_bind_tick", "b200_sixdof_tick",
    "b200_sixdof_trajectory_len", "b200_sixdof_trajectory_width", "b200_sixdof_trajectory_download",
    "b200_sixdof_trajectory_reset",
    "b200_sixdof_tick_count", "b200_sixdof_set_stream", "b200_sixdof_timings", "b200_sixdof_status",
    "b200_sixdof_device_plane", "b200_sixdof_plane_stride", "b200_probe_copy_gbs", "b200_probe_fp64_gflops",
    "b200_comm_available", "b200_comm_version", "b200_comm_unique_id", "b200_comm_create", "b200_comm_destroy",
    "b200_comm_rank", "b200_comm_size", "b200_comm_last_ms", "b200_sixdof_trajectory_gather_bytes",
    "b200_sixdof_trajectory_allgather", "b200_sixdof_step_row_sharded", "b200_probe_pcie_gbs",
    "b200_comm_peer_attach", "b200_comm_peer_attached", "b200_comm_peer_detach", "b200_selftest_shared_divisor", "b200_probe_zero_copy_gbs", "b200_egm08_stream_len", "b200_egm08_stream",
]
COMM_ID_BYTES = 128


class Effector(C.Structure):
    _fields_ = [
        ("kind", C.c_uint32),
        ("flags", C.c_uint32),
        ("p", C.c_double * 8),
        ("column_id", C.c_uint64),
        ("column_width", C.c_uint32),
        ("reserved", C.c_uint32),
        ("n_edges", C.c_uint64),
        ("edge_from", C.c_void_p),
        ("edge_to", C.c_void_p),
        ("entity_mask", C.c_void_p),
        ("table0", C.c_void_p),
        ("table1", C.c_void_p),
        ("table_len", C.c_uint64),
    ]


class Desc(C.Structure):
    _fields_ = [
        ("abi_version", C.c_uint32),
        ("integrator", C.c_uint32),
        ("math_mode", C.c_uint32),
        ("n_effectors", C.c_uint32),
        ("n_entities", C.c_uint64),
        ("n_worlds", C.c_uint64),
        ("sim_time_step", C.c_double),
        ("time_step", C.c_double),
        ("effectors", C.POINTER(Effector)),
        ("device", C.c_int32),
        ("max_fused_ticks", C.c_uint32),
        ("trajectory_every", C.c_uint32),
        ("invoke_chunk_bodies", C.c_uint32),
        ("trajectory_capacity", C.c_uint64),
        ("trajectory_flags", C.c_uint32),
        ("reserved0", C.c_uint32),
    ]


class Timings(C.Structure):
    _fields_ = [
        ("h2d_upload_ms", C.c_double),
        ("kernel_invoke_ms", C.c_double),
        ("d2h_download_ms", C.c_double),
        ("invoke_wall_ms", C.c_double),
        ("kernel_launches", C.c_uint64),
        ("ticks", C.c_uint64),
    ]


class B200Error(RuntimeError):
    """Backend failure (maps the reference's Error -> PyErr table, error.rs:46-58)."""

    def __init__(self, code: int, message: str):
        super().__init__(message)
        self.code = code


class B200ValueError(B200Error, ValueError):
    """ComponentNotFound / ValueSizeMismatch map to ValueError in the reference."""


_lib = None


def lib():
    """Load libb200_sixdof.so.  Raises if the CUDA extension has not been built:
    the product path never falls back to a CPU implementation."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise B200Error(
            ERR_NO_DEVICE,
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(make -C elodin_b200/csrc).  elodin_b200 has no CPU fallback.",
        )
    L = C.CDLL(LIB_PATH)
    vp, u64, u32 = C.c_void_p, C.c_uint64, C.c_uint32
    L.b200_component_id.argtypes = [C.c_char_p]
    L.b200_component_id.restype = u64
    L.b200_last_error.restype = C.c_char_p
    L.b200_device_count.restype = C.c_int
    L.b200_host_alloc.argtypes = [u64]
    L.b200_host_alloc.restype = vp
    L.b200_host_alloc_local.argtypes = [u64, C.c_int]
    L.b200_host_alloc_local.restype = vp
    L.b200_device_numa_node.argtypes = [C.c_int]
    L.b200_device_numa_node.restype = C.c_int
    L.b200_host_node_of.argtypes = [vp]
    L.b200_host_node_of.restype = C.c_int
    L.b200_host_free.argtypes = [vp]
    L.b200_host_free.restype = None
    L.b200_sixdof_create.argtypes = [C.POINTER(Desc), C.POINTER(vp)]
    L.b200_sixdof_destroy.argtypes = [vp]
    L.b200_sixdof_destroy.restype = None
    L.b200_sixdof_input_ids.argtypes = [vp, C.POINTER(u64), u32]
    L.b200_sixdof_input_ids.restype = u32
    L.b200_sixdof_output_ids.argtypes = [vp, C.POINTER(u64), u32]
    L.b200_sixdof_output_ids.restype = u32
    L.b200_sixdof_column_bytes.argtypes = [vp, u64]
    L.b200_sixdof_column_bytes.restype = u64
    L.b200_sixdof_upload.argtypes = [vp, u64, vp, u64]
    L.b200_sixdof_download.argtypes = [vp, u64, vp, u64]
    L.b200_sixdof_set_schedule.argtypes = [vp, u64, vp, u64, u64, u64]
    L.b200_sixdof_clear_schedule.argtypes = [vp, u64]
    L.b200_sixdof_step.argtypes = [vp, u64]
    L.b200_sixdof_sync.argtypes = [vp]
    L.b200_sixdof_invoke_batch.argtypes = [vp, C.POINTER(vp), C.POINTER(vp), u64]
    L.b200_sixdof_bind_tick.argtypes = [vp]
    L.b200_sixdof_tick.argtypes = [C.POINTER(vp), C.POINTER(vp)]
    L.b200_sixdof_tick.restype = None
    L.b200_sixdof_trajectory_len.argtypes = [vp]
    L.b200_sixdof_trajectory_len.restype = u64
    L.b200_sixdof_trajectory_width.argtypes = [vp]
    L.b200_sixdof_trajectory_width.restype = C.c_uint32
    L.b200_sixdof_trajectory_download.argtypes = [vp, vp, u64]
    L.b200_sixdof_trajectory_reset.argtypes = [vp]
    L.b200_sixdof_tick_count.argtypes = [vp]
    L.b200_sixdof_tick_count.restype = u64
    L.b200_sixdof_set_stream.argtypes = [vp, vp, C.c_int]
    L.b200_sixdof_timings.argtypes = [vp, C.POINTER(Timings)]
    L.b200_sixdof_status.argtypes = [vp]
    L.b200_sixdof_device_plane.argtypes = [vp, u64, u32]
    L.b200_sixdof_device_plane.restype = vp
    L.b200_sixdof_plane_stride.argtypes = [vp]
    L.b200_sixdof_plane_stride.restype = u64
    L.b200_comm_available.restype = C.c_int
    L.b200_comm_version.restype = C.c_int
    L.b200_comm_unique_id.argtypes = [vp, u32]
    L.b200_comm_create.argtypes = [vp, C.c_int, C.c_int, C.c_int, C.POINTER(vp)]
    L.b200_comm_destroy.argtypes = [vp]
    L.b200_comm_destroy.restype = None
    L.b200_comm_rank.argtypes = [vp]
    L.b200_comm_size.argtypes = [vp]
    L.b200_comm_last_ms.argtypes = [vp]
    L.b200_comm_last_ms.restype = C.c_double
    L.b200_sixdof_trajectory_gather_bytes.argtypes = [vp, C.POINTER(u64), C.c_int]
    L.b200_sixdof_trajectory_gather_bytes.restype = u64
    L.b200_sixdof_trajectory_allgather.argtypes = [vp, vp, C.POINTER(u64), vp, u64]
    L.b200_sixdof_step_row_sharded.argtypes = [vp, vp, u64]
    L.b200_egm08_stream_len.argtypes = [u32]
    L.b200_egm08_stream_len.restype = u64
    L.b200_egm08_stream.argtypes = [u32, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_double), u64]
    L.b200_selftest_shared_divisor.argtypes = [C.c_int, u64, u64, C.POINTER(u64)]
    L.b200_probe_zero_copy_gbs.argtypes = [C.c_int, vp, u64, u64, C.c_int, C.c_int, C.POINTER(C.c_double)]
    L.b200_comm_peer_attach.argtypes = [vp, vp]
    L.b200_comm_peer_attached.argtypes = [vp]
    L.b200_comm_peer_detach.argtypes = [vp]
    L.b200_comm_peer_detach.restype = None
    L.b200_probe_pcie_gbs.argtypes = [C.c_int, vp, u64, u64, C.c_int, C.POINTER(C.c_double)]
    L.b200_probe_copy_gbs.argtypes = [C.c_int, u64, C.c_int]
    L.b200_probe_copy_gbs.restype = C.c_double
    L.b200_probe_fp64_gflops.argtypes = [C.c_int, C.c_int]
    L.b200_probe_fp64_gflops.restype = C.c_double
    _lib = L
    return L


def check(rc: int) -> None:
    if rc == OK:
        return
    msg = lib().b200_last_error().decode("utf-8", "replace")
    if rc in (ERR_COMPONENT_NOT_FOUND, ERR_VALUE_SIZE_MISMATCH):
        raise B200ValueError(rc, msg)
    raise B200Error(rc, msg)


def component_id(name: str) -> int:
    """ComponentId::new (libs/impeller2/src/types.rs:40-45) — computed on the host
    in pure Python so metadata code works without loading the CUDA library."""
    h = 0xCBF29CE484222325
    for b in name.encode():
        h ^= b
        h = (h * 0x100000001B3) & 0xFFFFFFFFFFFFFFFF
    return h & ~(1 << 63)
