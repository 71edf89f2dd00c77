"""B200Exec — host-side mirror of the reference executor seam.

Reference: `CraneliftExec` / `WorldExec` (libs/nox-py/src/cranelift_exec.rs:13-195,
libs/nox-py/src/exec.rs:53-94).  Same contract: `invoke_batch(columns, n)` takes
the host column buffers (one per input ComponentId), integrates n ticks, and
returns every output column — but the state lives in B200 HBM between calls and
the ticks run in hand-written sm_100a kernels behind the C ABI
(include/b200_sixdof.h).  All numerics happen in libb200_sixdof.so.
"""

from __future__ import annotations

import ctypes as C
import math
from typing import Dict, Optional, Sequence

import numpy as np

from . import _lib
from ._lib import component_id

WORLD_POS = component_id("world_pos")
WORLD_VEL = component_id("world_vel")
WORLD_ACCEL = component_id("world_accel")
FORCE = component_id("force")
INERTIA = component_id("inertia")
TICK = component_id("tick")
SIMULATION_TIME_STEP = component_id("simulation_time_step")

_WIDTHS = {WORLD_POS: 7, WORLD_VEL: 6, WORLD_ACCEL: 6, FORCE: 6, INERTIA: 7}


def _cid(c) -> int:
    return component_id(c) if isinstance(c, str) else int(c)


class B200Exec:
    """One executor = one world batch ([n_worlds, n_entities] bodies) on one GPU."""

    def __init__(
        self,
        n_entities: int,
        n_worlds: int = 1,
        sim_time_step: float = 1.0 / 120.0,
        time_step: Optional[float] = None,
        effectors: Optional[Sequence] = None,
        integrator: str = "rk4",
        math: str = "exact",
        device: int = -1,
        max_fused_ticks: int = 1,
        trajectory_every: int = 0,
        trajectory_capacity: int = 0,
        world=None,
        invoke_chunk_bodies: int = 0,
        trajectory_full: bool = False,
    ):
        from .effectors import _flatten

        L = _lib.lib()
        effs = []
        for e in (effectors if isinstance(effectors, (list, tuple)) else _flatten(effectors)):
            effs += _flatten(e)
        if len(effs) > _lib.MAX_EFFECTORS:
            raise _lib.B200Error(_lib.ERR_UNSUPPORTED, f"too many effectors ({len(effs)} > {_lib.MAX_EFFECTORS})")
        self._effector_objs = effs
        arr = (_lib.Effector * max(len(effs), 1))()
        self._column_widths: Dict[int, int] = dict(_WIDTHS)
        for i, e in enumerate(effs):
            arr[i] = e.lower(world)
            if arr[i].column_id:
                self._column_widths[int(arr[i].column_id)] = int(arr[i].column_width)
        d = _lib.Desc()
        d.abi_version = _lib.ABI_VERSION
        d.integrator = {"rk4": _lib.INTEGRATOR_RK4, "semi_implicit": _lib.INTEGRATOR_SEMI_IMPLICIT}[integrator]
        d.math_mode = {"exact": _lib.MATH_EXACT, "fast": _lib.MATH_FAST}[math]
        d.n_effectors = len(effs)
        d.n_entities, d.n_worlds = int(n_entities), int(n_worlds)
        d.sim_time_step = float(sim_time_step)
        d.time_step = math_nan() if time_step is None else float(time_step)
        d.effectors = arr
        d.device = int(device)
        d.max_fused_ticks = int(max_fused_ticks)
        d.trajectory_every = int(trajectory_every)
        d.trajectory_capacity = int(trajectory_capacity)
        d.invoke_chunk_bodies = int(invoke_chunk_bodies)
        d.trajectory_flags = _lib.TRAJ_FULL if trajectory_full else 0
        h = C.c_void_p()
        _lib.check(L.b200_sixdof_create(C.byref(d), C.byref(h)))
        self._L, self._h = L, h
        self.n_entities, self.n_worlds = int(n_entities), int(n_worlds)
        self.integrator, self.math = integrator, math
        ids = (C.c_uint64 * 32)()
        n = L.b200_sixdof_input_ids(h, ids, 32)
        self.input_ids = [int(ids[i]) for i in range(n)]
        n = L.b200_sixdof_output_ids(h, ids, 32)
        self.output_ids = [int(ids[i]) for i in range(n)]

    # ---- lifetime -------------------------------------------------------------
    def close(self) -> None:
        if getattr(self, "_h", None):
            self._L.b200_sixdof_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    # ---- metadata -------------------------------------------------------------
    def column_bytes(self, cid) -> int:
        return int(self._L.b200_sixdof_column_bytes(self._h, _cid(cid)))

    def column_shape(self, cid):
        cid = _cid(cid)
        if cid in (TICK, SIMULATION_TIME_STEP):
            return (1,)
        return (self.n_worlds, self.n_entities, self._column_widths[cid])

    @property
    def tick(self) -> int:
        return int(self._L.b200_sixdof_tick_count(self._h))

    # ---- data movement ----------------------------------------------------------
    def upload(self, cid, array) -> None:
        cid = _cid(cid)
        dtype = np.uint64 if cid == TICK else np.float64
        a = np.ascontiguousarray(array, dtype=dtype)
        _lib.check(self._L.b200_sixdof_upload(self._h, cid, a.ctypes.data, a.nbytes))
        # the copy out of `a` is asynchronous on the handle's stream
        _lib.check(self._L.b200_sixdof_sync(self._h))

    def upload_ptr(self, cid, ptr: int, nbytes: int) -> None:
        """Upload from a raw host or device pointer (e.g. a torch tensor's data_ptr())."""
        _lib.check(self._L.b200_sixdof_upload(self._h, _cid(cid), C.c_void_p(ptr), nbytes))

    def download(self, cid, out: Optional[np.ndarray] = None) -> np.ndarray:
        cid = _cid(cid)
        dtype = np.uint64 if cid == TICK else np.float64
        if out is None:
            out = np.empty(self.column_shape(cid), dtype=dtype)
        _lib.check(self._L.b200_sixdof_download(self._h, cid, out.ctypes.data, out.nbytes))
        return out

    def download_ptr(self, cid, ptr: int, nbytes: int) -> None:
        _lib.check(self._L.b200_sixdof_download(self._h, _cid(cid), C.c_void_p(ptr), nbytes))

    def set_state(self, pos=None, vel=None, inertia=None, accel=None, force=None, **columns) -> None:
        for cid, a in ((WORLD_POS, pos), (WORLD_VEL, vel), (INERTIA, inertia), (WORLD_ACCEL, accel), (FORCE, force)):
            if a is not None:
                self.upload(cid, a)
        for name, a in columns.items():
            self.upload(name, a)

    # ---- input schedules ----------------------------------------------------------
    def set_schedule(self, cid, rows, first_tick: int = 0) -> None:
        """Drive effector input column `cid` from per-tick rows held on the device: `rows` is
        [T, n_worlds, n_entities, width]; the tick whose Tick value is k reads row clamp(k - first_tick, 0, T - 1).
        Replaces an earlier schedule of the column.  See b200_sixdof_set_schedule."""
        cid = _cid(cid)
        a = np.ascontiguousarray(rows, dtype=np.float64)
        if a.ndim != 4 or a.shape[0] < 1:
            raise _lib.B200ValueError(_lib.ERR_VALUE_SIZE_MISMATCH,
                                      f"schedule rows must be [T >= 1, n_worlds, n_entities, width], got shape {a.shape}")
        if first_tick < 0:
            raise ValueError(f"first_tick must be >= 0, got {first_tick}")
        _lib.check(self._L.b200_sixdof_set_schedule(self._h, cid, a.ctypes.data, a.nbytes, a.shape[0], int(first_tick)))

    def clear_schedule(self, cid) -> None:
        """Unbind the schedule of `cid`: the column keeps the row its last tick used, later ticks read the column."""
        _lib.check(self._L.b200_sixdof_clear_schedule(self._h, _cid(cid)))

    # ---- stepping ---------------------------------------------------------------
    def step(self, n_ticks: int = 1, sync: bool = False) -> None:
        _lib.check(self._L.b200_sixdof_step(self._h, int(n_ticks)))
        if sync:
            self.sync()

    def sync(self) -> None:
        _lib.check(self._L.b200_sixdof_sync(self._h))

    def invoke_batch(self, in_cols: Sequence[np.ndarray], n_ticks: int = 1,
                     out_cols: Optional[Sequence[np.ndarray]] = None):
        """CraneliftExec::invoke_batch (cranelift_exec.rs:129-195): `in_cols[i]` is the
        host buffer of `input_ids[i]` (None: not dirty; always None for a scheduled column);
        returns the buffers of `output_ids`."""
        if len(in_cols) != len(self.input_ids):
            raise _lib.B200ValueError(_lib.ERR_VALUE_SIZE_MISMATCH, "wrong number of input columns")
        ins = []
        for cid, a in zip(self.input_ids, in_cols):
            if a is None:  # not dirty: the device-resident copy stands (world.rs:43,249-252)
                ins.append(None)
                continue
            a = np.ascontiguousarray(a, dtype=np.uint64 if cid == TICK else np.float64)
            if a.nbytes != self.column_bytes(cid):
                raise _lib.B200ValueError(_lib.ERR_VALUE_SIZE_MISMATCH, "value size mismatch")
            ins.append(a)
        if out_cols is None:
            out_cols = [np.empty(self.column_shape(cid), dtype=np.uint64 if cid == TICK else np.float64)
                        for cid in self.output_ids]
        elif len(out_cols) != len(self.output_ids):
            raise _lib.B200ValueError(_lib.ERR_VALUE_SIZE_MISMATCH, "wrong number of output columns")
        in_ptrs = (C.c_void_p * len(ins))(*[None if a is None else a.ctypes.data for a in ins])
        out_ptrs = (C.c_void_p * len(out_cols))(*[None if a is None else a.ctypes.data for a in out_cols])
        _lib.check(self._L.b200_sixdof_invoke_batch(self._h, in_ptrs, out_ptrs, int(n_ticks)))
        return list(out_cols)

    def invoke_batch_ptrs(self, in_ptrs: Sequence[Optional[int]], out_ptrs: Sequence[Optional[int]], n_ticks: int) -> None:
        """Raw-pointer form.  A None / 0 input = "not dirty" (the device-resident copy stands, world.rs:43,249-252);
        a None / 0 output = not read back after this batch."""
        ip = (C.c_void_p * len(in_ptrs))(*in_ptrs)
        op = (C.c_void_p * len(out_ptrs))(*out_ptrs)
        _lib.check(self._L.b200_sixdof_invoke_batch(self._h, ip, op, int(n_ticks)))

    def tick_fn(self, in_cols: Sequence[np.ndarray], out_cols: Sequence[np.ndarray]) -> None:
        """The TickFn-shaped entry (cranelift_exec.rs:11): one tick, void return."""
        _lib.check(self._L.b200_sixdof_bind_tick(self._h))
        ip = (C.c_void_p * len(in_cols))(*[a.ctypes.data for a in in_cols])
        op = (C.c_void_p * len(out_cols))(*[a.ctypes.data for a in out_cols])
        self._L.b200_sixdof_tick(ip, op)
        _lib.check(self._L.b200_sixdof_status(self._h))

    # ---- trajectory ---------------------------------------------------------------
    def trajectory_len(self) -> int:
        return int(self._L.b200_sixdof_trajectory_len(self._h))

    def trajectory_width(self) -> int:
        """13 = (world_pos[7], world_vel[6]); 25 with trajectory_full: + (world_accel[6], force[6])."""
        return int(self._L.b200_sixdof_trajectory_width(self._h))

    def trajectory(self) -> np.ndarray:
        """[samples, n_worlds, n_entities, width] — see trajectory_width()."""
        self.sync()
        n = self.trajectory_len()
        out = np.empty((n, self.n_worlds, self.n_entities, max(self.trajectory_width(), 13)))
        _lib.check(self._L.b200_sixdof_trajectory_download(self._h, out.ctypes.data, out.nbytes))
        return out

    def trajectory_to_ptr(self, ptr: int, nbytes: int) -> None:
        _lib.check(self._L.b200_sixdof_trajectory_download(self._h, C.c_void_p(ptr), nbytes))

    def trajectory_reset(self) -> None:
        _lib.check(self._L.b200_sixdof_trajectory_reset(self._h))

    # ---- plumbing ---------------------------------------------------------------
    def set_stream(self, cuda_stream: Optional[int]) -> None:
        """Run on a caller-owned cudaStream_t (0 = the legacy default stream, which is what
        torch.cuda.current_stream().cuda_stream returns by default); None = private stream."""
        if cuda_stream is None:
            _lib.check(self._L.b200_sixdof_set_stream(self._h, C.c_void_p(0), 1))
        else:
            _lib.check(self._L.b200_sixdof_set_stream(self._h, C.c_void_p(int(cuda_stream)), 0))

    def timings(self) -> dict:
        t = _lib.Timings()
        _lib.check(self._L.b200_sixdof_timings(self._h, C.byref(t)))
        return {"h2d_upload_ms": t.h2d_upload_ms, "kernel_invoke_ms": t.kernel_invoke_ms,
                "d2h_download_ms": t.d2h_download_ms, "invoke_wall_ms": t.invoke_wall_ms,
                "kernel_launches": int(t.kernel_launches),
                "ticks": int(t.ticks)}

    def device_plane(self, cid, plane: int) -> int:
        return int(self._L.b200_sixdof_device_plane(self._h, _cid(cid), plane) or 0)

    @property
    def plane_stride(self) -> int:
        return int(self._L.b200_sixdof_plane_stride(self._h))


def math_nan() -> float:
    return math.nan


def device_count() -> int:
    n = _lib.lib().b200_device_count()
    return max(int(n), 0)


def pinned_empty(shape, dtype=np.float64, device: Optional[int] = None) -> np.ndarray:
    """numpy array over page-locked host memory (b200_host_alloc); with `device`, on the NUMA node of that
    GPU's PCIe root (b200_host_alloc_local)."""
    L = _lib.lib()
    dtype = np.dtype(dtype)
    n = int(np.prod(shape)) * dtype.itemsize
    p = L.b200_host_alloc(max(n, 1)) if device is None else L.b200_host_alloc_local(max(n, 1), int(device))
    if not p:
        raise _lib.B200Error(_lib.ERR_OUT_OF_MEMORY, L.b200_last_error().decode())
    buf = (C.c_char * max(n, 1)).from_address(p)
    arr = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)
    _PINNED[arr.ctypes.data] = p
    return arr


_PINNED: Dict[int, int] = {}


def pinned_free(arr: np.ndarray) -> None:
    p = _PINNED.pop(arr.ctypes.data, None)
    if p:
        _lib.lib().b200_host_free(C.c_void_p(p))
