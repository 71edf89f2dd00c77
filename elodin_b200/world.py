"""Host-side mirror of the nox-py ECS surface for the six_dof() path.

Reference (what each piece mirrors):
  * spatial value types          libs/nox-py/src/spatial.rs, libs/nox/src/spatial.rs
  * Component / Archetype / Body python/elodin/__init__.py:594-669, six_dof.rs:153-159
  * World (host columns)         libs/nox-py/src/world.rs:25-60,174-200
  * WorldBuilder.build / run     libs/nox-py/src/world_builder.rs:550-720,1737-1775
  * Exec.run / history           libs/nox-py/src/exec.rs:104-173
  * six_dof(), Integrator        libs/nox-py/src/lib.rs:106-127, six_dof.rs:161-203

Only data handling lives here (numpy host columns, entity/component indexing,
tick bookkeeping).  Every tick is integrated by libb200_sixdof.so on the GPU via
B200Exec; there is no Python/CPU integrator in this package.
"""

from __future__ import annotations

import dataclasses
import enum
import re
import copy
import os
import sys
import time
import typing
from typing import Callable, Dict, List, Optional, Sequence, Union

import numpy as np

from . import _lib
from ._lib import component_id
from .effectors import Effector, System, _flatten
from .executor import B200Exec

# --------------------------------------------------------------------------- value types


def _vec(x, n) -> np.ndarray:
    a = np.zeros(n) if x is None else np.asarray(x, dtype=np.float64).reshape(n)
    return a


class Quaternion:
    """[i, j, k, w] storage, scalar last (libs/nox/src/quaternion.rs:100)."""

    def __init__(self, arr):
        self.arr = _vec(arr, 4)

    @staticmethod
    def identity() -> "Quaternion":
        return Quaternion([0.0, 0.0, 0.0, 1.0])

    @staticmethod
    def from_axis_angle(axis, angle) -> "Quaternion":
        axis = np.asarray(axis, dtype=np.float64)
        axis = axis / np.sqrt(axis @ axis)
        half = angle / 2.0
        return Quaternion(np.concatenate([axis * np.sin(half), [np.cos(half)]]))

    @staticmethod
    def from_euler(angles) -> "Quaternion":
        """roll, pitch, yaw — libs/nox/src/quaternion.rs:105-124."""
        r, p, y = [float(a) for a in angles]
        cr, sr, cp, sp, cy, sy = (np.cos(r / 2), np.sin(r / 2), np.cos(p / 2), np.sin(p / 2), np.cos(y / 2),
                                  np.sin(y / 2))
        return Quaternion([sr * cp * cy - cr * sp * sy, cr * sp * cy + sr * cp * sy, cr * cp * sy - sr * sp * cy,
                           cr * cp * cy + sr * sp * sy])

    def vector(self) -> np.ndarray:
        return self.arr


class SpatialTransform:
    """7 f64: [q(4), x(3)] (libs/nox/src/spatial.rs:14)."""

    WIDTH = 7

    def __init__(self, arr=None, angular: Optional[Quaternion] = None, linear=None):
        if arr is not None:
            if angular is not None or linear is not None:
                raise ValueError("Cannot specify both array and linear/angular")
            self.arr = _vec(arr, 7)
        else:
            q = angular.arr if angular is not None else Quaternion.identity().arr
            self.arr = np.concatenate([q, _vec(linear, 3)])

    def linear(self):
        return self.arr[4:]

    def angular(self) -> Quaternion:
        return Quaternion(self.arr[:4])

    def asarray(self):
        return self.arr


class SpatialMotion:
    """6 f64: [angular(3), linear(3)] (libs/nox/src/spatial.rs:386,432-436)."""

    WIDTH = 6

    def __init__(self, angular=None, linear=None):
        self.arr = np.concatenate([_vec(angular, 3), _vec(linear, 3)])

    def linear(self):
        return self.arr[3:]

    def angular(self):
        return self.arr[:3]

    def asarray(self):
        return self.arr


class SpatialForce:
    """6 f64: [torque(3), force(3)] (libs/nox/src/spatial.rs:141,207-211)."""

    WIDTH = 6

    def __init__(self, arr=None, torque=None, linear=None):
        self.arr = _vec(arr, 6) if arr is not None else np.concatenate([_vec(torque, 3), _vec(linear, 3)])

    def force(self):
        return self.arr[3:]

    def torque(self):
        return self.arr[:3]

    def asarray(self):
        return self.arr


class SpatialInertia:
    """7 f64: [diag(3), momentum(3), mass]; `SpatialInertia(mass)` sets diag = mass
    (libs/nox-py/src/spatial.rs:385-397, libs/nox/src/spatial.rs:315-338)."""

    WIDTH = 7

    def __init__(self, mass, inertia=None):
        mass = float(mass)
        diag = np.ones(3) * mass if inertia is None else _vec(inertia, 3)
        self.arr = np.concatenate([diag, np.zeros(3), [mass]])

    def mass(self):
        return self.arr[6]

    def inertia_diag(self):
        return self.arr[:3]

    def asarray(self):
        return self.arr


# --------------------------------------------------------------------------- components


class PrimitiveType(enum.Enum):
    F64 = "f64"
    U64 = "u64"


class ComponentType:
    def __init__(self, ty: PrimitiveType = PrimitiveType.F64, shape: Sequence[int] = ()):
        self.ty, self.shape = ty, tuple(shape)

    @property
    def width(self) -> int:
        return int(np.prod(self.shape)) if self.shape else 1


ComponentType.F64 = ComponentType(PrimitiveType.F64, ())
ComponentType.U64 = ComponentType(PrimitiveType.U64, ())
ComponentType.SpatialPosF64 = ComponentType(PrimitiveType.F64, (7,))
ComponentType.SpatialMotionF64 = ComponentType(PrimitiveType.F64, (6,))
ComponentType.Edge = ComponentType(PrimitiveType.U64, (2,))


class Component:
    """`Component(name, ty, metadata=...)` — python/elodin/__init__.py Annotated metadata;
    id = FNV-1a (libs/impeller2/src/types.rs:40-45)."""

    def __init__(self, name: str, ty: Optional[ComponentType] = None, metadata: Optional[dict] = None):
        self.name, self.ty, self.metadata = name, ty, metadata or {}

    @property
    def id(self) -> int:
        return component_id(self.name)

    @staticmethod
    def of(annotated) -> "Component":
        for m in getattr(annotated, "__metadata__", ()):
            if isinstance(m, Component):
                return m
        raise TypeError(f"{annotated!r} carries no Component metadata")


Annotated = typing.Annotated

WorldPos = Annotated[SpatialTransform, Component("world_pos", ComponentType.SpatialPosF64,
                                                 {"element_names": "q0,q1,q2,q3,x,y,z", "priority": 5})]
WorldVel = Annotated[SpatialMotion, Component("world_vel", ComponentType.SpatialMotionF64,
                                              {"element_names": "ωx,ωy,ωz,x,y,z", "priority": 5})]
WorldAccel = Annotated[SpatialMotion, Component("world_accel", ComponentType.SpatialMotionF64,
                                                {"element_names": "αx,αy,αz,x,y,z", "priority": 5})]
Force = Annotated[SpatialForce, Component("force", ComponentType.SpatialMotionF64,
                                          {"element_names": "τx,τy,τz,x,y,z", "priority": 5})]
Inertia = Annotated[SpatialInertia, Component("inertia", ComponentType(PrimitiveType.F64, (7,)), {"priority": 5})]
Seed = Annotated[np.ndarray, Component("seed", ComponentType.U64, {"priority": 5})]
SimulationTick = Annotated[np.ndarray, Component("tick", ComponentType.F64, {"priority": 7})]
SimulationTimeStep = Annotated[np.ndarray, Component("simulation_time_step", ComponentType.F64, {"priority": 8})]


class Edge:
    """Directed edge between two entities (GraphQuery edges)."""

    def __init__(self, left: "EntityId", right: "EntityId"):
        self.left, self.right = EntityId(int(left)), EntityId(int(right))


class EntityId(int):
    pass


_snake = re.compile(r"(?<!^)(?=[A-Z])")


class Archetype:
    """Dataclass whose fields are Annotated[..., Component(...)] (reference Archetype)."""

    @classmethod
    def archetype_name(cls) -> str:
        return _snake.sub("_", cls.__name__).lower()

    def component_values(self) -> List[tuple]:
        hints = typing.get_type_hints(type(self), include_extras=True)
        out = []
        for f in dataclasses.fields(self):  # type: ignore[arg-type]
            comp = Component.of(hints[f.name])
            out.append((comp, getattr(self, f.name)))
        return out


def dataclass(cls):
    return dataclasses.dataclass(cls)


@dataclasses.dataclass
class Body(Archetype):
    """python/elodin/__init__.py:664-669."""

    world_pos: WorldPos = dataclasses.field(default_factory=SpatialTransform)
    world_vel: WorldVel = dataclasses.field(default_factory=SpatialMotion)
    inertia: Inertia = dataclasses.field(default_factory=lambda: SpatialInertia(mass=1.0))
    force: Force = dataclasses.field(default_factory=SpatialForce)
    world_accel: WorldAccel = dataclasses.field(default_factory=SpatialMotion)


def _flat(value) -> np.ndarray:
    if isinstance(value, Edge):
        return np.array([int(value.left), int(value.right)], dtype=np.uint64)
    if hasattr(value, "asarray"):
        return np.asarray(value.asarray(), dtype=np.float64).reshape(-1)
    return np.atleast_1d(np.asarray(value)).reshape(-1)


# --------------------------------------------------------------------------- systems


class Integrator(enum.Enum):
    Rk4 = "rk4"
    SemiImplicit = "semi_implicit"


@dataclasses.dataclass
class SixDof(System):
    time_step: Optional[float]
    effectors: list
    integrator: Integrator


def six_dof(time_step: Optional[float] = None, sys: Optional[System] = None,
            integrator: Integrator = Integrator.Rk4) -> SixDof:
    """`el.six_dof(time_step=None, sys=None, integrator=Integrator.Rk4)` (lib.rs:106-127):
    clear_forces | sys | calc_accel under the chosen integrator (six_dof.rs:161-203)."""
    return SixDof(time_step, _flatten(sys), integrator)


@dataclasses.dataclass
class HostSystem(System):
    """A per-tick host callback over the numpy columns (non-effector systems such as
    the rocket's thrust curve, examples/rocket/main.py:416-426).  It runs on the host
    between GPU ticks, like copy_db_to_world feeding external controls
    (impeller2_server.rs:607), and forces one tick per launch.  An input known ahead of
    time and indexed by tick (a thrust curve) runs faster as an input_schedule()."""

    fn: Callable[["StepContext"], None]


def host_system(fn) -> HostSystem:
    return HostSystem(fn)


@dataclasses.dataclass(eq=False)
class InputSchedule(System):
    """Per-tick rows of an effector input column, held on the device (B200Exec.set_schedule): a thrust curve, a
    recorded wind or a per-world open-loop profile without a host callback, so the run keeps the device-resident
    route and fused ticks."""

    component: str
    rows: np.ndarray
    first_tick: int = 0


def input_schedule(component, rows, first_tick: int = 0) -> InputSchedule:
    """`el.input_schedule("thrust", rows, first_tick=0) | el.six_dof(...)`: the tick whose Tick value is k sees
    row clamp(k - first_tick, 0, T - 1) in the effector input column `component` — the same values a host_system
    writing `rows[tick]` before every tick would leave there.  `rows` is [T, n_owner_entities(, width)] (one curve
    for every world) or [T, n_worlds, n_owner_entities, width]; owner entities are the ones that carry the component,
    in spawn order."""
    if isinstance(component, Component):
        name = component.name
    elif isinstance(component, str):
        name = component
    else:
        name = Component.of(component).name
    if int(first_tick) < 0:
        raise ValueError(f"input_schedule({name!r}): first_tick must be >= 0, got {first_tick}")
    return InputSchedule(name, np.asarray(rows, dtype=np.float64), int(first_tick))


def schedule_row(tick, first_tick: int, n_rows: int):
    """Row of an input schedule that the tick whose Tick value is `tick` reads (scalar or array of ticks); the rule
    of b200_sixdof_set_schedule."""
    return np.clip(np.asarray(tick, dtype=np.int64) - int(first_tick), 0, int(n_rows) - 1)


def _schedule_rows(name: str, rows: np.ndarray, n_worlds: int, n_owner: int, width: int) -> np.ndarray:
    """[T, n_worlds, n_owner, width] from the shapes input_schedule accepts (broadcast over worlds on the host)."""
    a = np.asarray(rows, dtype=np.float64)
    if a.ndim == 2 and width == 1:
        a = a[:, :, None]
    if a.ndim == 3 and a.shape[1:] == (n_owner, width):
        a = np.broadcast_to(a[:, None], (a.shape[0], n_worlds, n_owner, width))
    elif not (a.ndim == 4 and a.shape[1:] == (n_worlds, n_owner, width)):
        want = f"[T, {n_owner}, {width}] or [T, {n_worlds}, {n_owner}, {width}]" + (f" or [T, {n_owner}]" if width == 1 else "")
        raise ValueError(f"input_schedule({name!r}): rows of shape {a.shape}, expected {want}")
    if a.shape[0] < 1:
        raise ValueError(f"input_schedule({name!r}): the schedule needs at least one row")
    return np.ascontiguousarray(a)


class StepContext:
    def __init__(self, exec_: "Exec"):
        self._exec = exec_

    @property
    def tick(self) -> int:
        return self._exec.tick

    def _unscheduled(self, name: str) -> int:
        cid = component_id(name)
        if cid in self._exec._schedules:
            raise ValueError(f"column '{name}' is driven by an input_schedule: a host system cannot read or write it")
        return cid

    def column(self, name: str) -> np.ndarray:
        """[n_worlds, n_entities_with_component, width] numpy view of a host column."""
        cid = self._unscheduled(name)
        return self._exec.world.columns[cid].buffer

    def write_component(self, pair_name: str, value) -> None:
        ent, comp = pair_name.rsplit(".", 1)
        cid = self._unscheduled(comp)
        col = self._exec.world.columns[cid]
        row = col.row_of(self._exec.world.entity_by_name(ent))
        col.buffer[:, row, :] = np.asarray(value, dtype=col.buffer.dtype).reshape(-1)
        self._exec.dirty.add(col.component.id)


# --------------------------------------------------------------------------- world


class Column:
    """`Column{buffer, entity_ids}` (world.rs:25-29) with a leading world axis."""

    def __init__(self, component: Component, width: int, dtype):
        self.component, self.width, self.dtype = component, width, dtype
        self.entity_ids: List[int] = []
        self.rows: List[np.ndarray] = []
        self.buffer: Optional[np.ndarray] = None

    def row_of(self, entity: int) -> int:
        return self.entity_ids.index(int(entity))


def quantised_time_step(simulation_rate: float) -> float:
    """`Duration::from_secs_f64(1/rate).as_secs_f64()` (world_builder.rs:221,
    world.rs:185-191): the step is rounded to whole nanoseconds; 120 Hz -> 0.008333333."""
    if simulation_rate <= 0:
        raise ValueError(f"simulation_rate must be > 0 Hz, got {simulation_rate}")
    ns = int(np.rint(1.0e9 / simulation_rate))
    secs, nanos = divmod(ns, 1_000_000_000)
    return float(secs) + float(nanos) / 1.0e9


def ticks_per_telemetry(simulation_rate: float, telemetry_rate: Optional[float]) -> int:
    """validate_rates, world_builder.rs:211-243."""
    if telemetry_rate is None:
        return 1
    if telemetry_rate <= 0:
        raise ValueError(f"telemetry_rate must be > 0 Hz, got {telemetry_rate}")
    ratio = simulation_rate / telemetry_rate
    rounded = round(ratio)
    if abs(ratio - rounded) > 1e-9 or rounded < 1:
        raise ValueError(
            f"telemetry_rate ({telemetry_rate} Hz) must evenly divide simulation_rate ({simulation_rate} Hz); got ratio {ratio}")
    return max(int(rounded), 1)


class World:
    """Host ECS world.  Entity 0 is `Globals` (tick, simulation_time_step), spawned on
    construction like World::add_globals (world.rs:174-183)."""

    def __init__(self):
        self.columns: Dict[int, Column] = {}
        self.entity_names: Dict[int, str] = {0: "Globals"}
        self.entity_len = 1
        self.edges: List[tuple] = []  # (component_name, from_entity, to_entity) in spawn order

    # -- spawning ---------------------------------------------------------------
    def spawn(self, archetypes, name: Optional[str] = None, id: Optional[str] = None) -> EntityId:
        ent = EntityId(self.entity_len)
        self.entity_len += 1
        if not isinstance(archetypes, (list, tuple)):
            archetypes = [archetypes]
        for arch in archetypes:
            for comp, value in arch.component_values():
                flat = _flat(value)
                if isinstance(value, Edge):
                    self.edges.append((comp.name, int(value.left), int(value.right)))
                col = self.columns.get(comp.id)
                if col is None:
                    col = Column(comp, len(flat), flat.dtype if flat.dtype == np.uint64 else np.float64)
                    self.columns[comp.id] = col
                if len(flat) != col.width:
                    raise _lib.B200ValueError(_lib.ERR_VALUE_SIZE_MISMATCH, "value size mismatch")
                col.entity_ids.append(int(ent))
                col.rows.append(flat.astype(col.dtype))
        if name is not None:
            self.entity_names[int(ent)] = name
        elif id is not None:
            self.entity_names[int(ent)] = id
        return ent

    def entity_by_name(self, name: str) -> int:
        for e, n in self.entity_names.items():
            if n == name or n.lower() == name:
                return e
        raise _lib.B200ValueError(_lib.ERR_COMPONENT_NOT_FOUND, f"entity not found: {name}")

    # -- queries ---------------------------------------------------------------
    def body_entities(self) -> List[int]:
        col = self.columns.get(component_id("world_pos"))
        return list(col.entity_ids) if col else []

    def edge_rows(self) -> np.ndarray:
        """Spawned edges as (from_row, to_row) pairs over the Body rows, spawn order kept."""
        rows = {e: i for i, e in enumerate(self.body_entities())}
        out = [(rows[a], rows[b]) for (_, a, b) in self.edges if a in rows and b in rows]
        return np.asarray(out, dtype=np.uint32).reshape(-1, 2)

    def _clone_for_exec(self) -> "World":
        """Private copy for one Exec: same entities / names / edges, its own Column objects and buffers."""
        w = copy.copy(self)
        w.columns = {}
        for cid, col in self.columns.items():
            c = Column(col.component, col.width, col.dtype)
            c.entity_ids = list(col.entity_ids)
            c.rows = [r.copy() for r in col.rows]
            c.buffer = None if col.buffer is None else col.buffer.copy()
            w.columns[cid] = c
        w.entity_names = dict(self.entity_names)
        w.edges = list(self.edges)
        return w

    def finalize(self, n_worlds: int = 1) -> None:
        for col in self.columns.values():
            base = np.stack(col.rows).astype(col.dtype) if col.rows else np.zeros((0, col.width), col.dtype)
            col.buffer = np.broadcast_to(base, (n_worlds,) + base.shape).copy()

    # -- build / run -------------------------------------------------------------
    def build(self, system: System, simulation_rate: float = 120.0, generate_real_time: bool = False,
              telemetry_rate: Optional[float] = None, default_playback_speed: float = 1.0,
              max_ticks: Optional[int] = None, optimize: bool = False, db_path: Optional[str] = None,
              backend: str = "b200", math: str = "exact", n_worlds: int = 1, device: int = -1,
              world_params: Optional[Dict[str, np.ndarray]] = None, resident: Optional[bool] = None) -> "Exec":
        if backend not in ("b200", "b200-exact", "b200-fast"):
            raise _lib.B200Error(
                _lib.ERR_UNSUPPORTED,
                f"unknown backend '{backend}': this package only provides 'b200' (no cranelift / jax fallback)")
        if backend == "b200-fast":
            math = "fast"
        return Exec(self, system, simulation_rate, telemetry_rate, max_ticks, math, n_worlds, device, world_params, resident)

    def run(self, system: System, simulation_rate: float = 120.0, generate_real_time: bool = False,
            telemetry_rate: Optional[float] = None, default_playback_speed: float = 1.0,
            max_ticks: Optional[int] = None, optimize: bool = False, is_canceled=None, pre_step=None,
            post_step=None, db_path: Optional[str] = None, interactive: bool = True, start_timestamp=None,
            log_level=None, backend: str = "b200", math: str = "exact", n_worlds: int = 1) -> "Exec":
        """Headless `World.run` (python/elodin/__init__.py:673-718): runs to max_ticks.  The
        DB server / editor layers of the reference are out of scope.  Like the reference's
        WorldBuilder::run it looks at sys.argv: `python sim.py bench --ticks N [--detail]`
        builds, runs N ticks and prints the reference's bench lines (world_builder.rs:868-909),
        which examples/n-body/benchmark_backends.py parses."""
        argv = sys.argv[1:]
        if argv[:1] == ["bench"]:
            ticks = int(argv[argv.index("--ticks") + 1]) if "--ticks" in argv else 1000
            t0 = time.perf_counter()
            ex = self.build(system, simulation_rate, generate_real_time, telemetry_rate, default_playback_speed,
                            max_ticks, optimize, db_path, backend, math, n_worlds)
            ex.build_ms = (time.perf_counter() - t0) * 1e3
            ex.run(ticks, show_progress=False)
            prof = ex.profile()
            tpt = int(prof["ticks_per_telemetry"])
            print(f"= tick time:          {prof['tick']:.3f} ms (batch of {tpt} ticks)")
            print(f"build time:           {prof['build']:.3f} ms")
            print(f"real_time_factor:     {prof['real_time_factor']:.3f}")
            if "--detail" in argv:
                print(f"copy_to_client time:  {prof['copy_to_client']:.3f} ms")
                print(f"execute_buffers time: {prof['execute_buffers']:.3f} ms")
                print(f"copy_to_host time:    {prof['copy_to_host']:.3f} ms")
                print(f"h2d_upload time:      {prof['h2d_upload']:.3f} ms")
                print(f"kernel_invoke time:   {prof['kernel_invoke']:.3f} ms ({tpt} invocations)")
                print(f"d2h_download time:    {prof['d2h_download']:.3f} ms")
                print(f"add_to_history time:  {prof['add_to_history']:.3f} ms")
            return ex
        if max_ticks is None:
            raise ValueError("elodin_b200.World.run is headless: pass max_ticks")
        ex = self.build(system, simulation_rate, generate_real_time, telemetry_rate, default_playback_speed,
                        max_ticks, optimize, db_path, backend, math, n_worlds)
        if db_path:
            # the reference's `World.run(db_path=...)` leaves an elodin-db directory behind (impeller2_server.rs:
            # 229-309, 390-438): init_db now, one commit per telemetry cycle while the run is in flight
            ts = None
            if start_timestamp is not None:
                ts = int(start_timestamp.timestamp() * 1e6) if hasattr(start_timestamp, "timestamp") else int(start_timestamp)
            ex.attach_db(db_path, ts)
        ex.run(max_ticks, show_progress=False, is_canceled=is_canceled, pre_step=pre_step, post_step=post_step)
        if db_path:
            ex.close_db()
        return ex


class _Row(np.ndarray):
    def to_numpy(self):
        return np.asarray(self)


class _Series(np.ndarray):
    """History rows; `[-1].to_numpy()` works like the reference's polars output."""

    def __getitem__(self, i):
        r = super().__getitem__(i)
        return r.view(_Row) if isinstance(r, np.ndarray) else r


class Exec:
    """`PyExec` (libs/nox-py/src/exec.rs:96-173): owns the world + a B200Exec."""

    def __init__(self, world: World, system: System, simulation_rate: float, telemetry_rate: Optional[float],
                 max_ticks: Optional[int], math: str, n_worlds: int, device: int,
                 world_params: Optional[Dict[str, np.ndarray]], resident: Optional[bool] = None):
        systems = _flatten(system)
        six = [s for s in systems if isinstance(s, SixDof)]
        if len(six) != 1:
            raise _lib.B200Error(_lib.ERR_UNSUPPORTED, "the B200 backend runs exactly one six_dof() system per world")
        self.six = six[0]
        pre = systems[: systems.index(self.six)]
        post = systems[systems.index(self.six) + 1:]
        for s in pre + post:
            if not isinstance(s, (HostSystem, InputSchedule)):
                raise _lib.B200Error(_lib.ERR_UNSUPPORTED,
                                     f"{s!r}: only host_system() callbacks may surround six_dof() (no tracing compiler)")
            if isinstance(s, InputSchedule) and s in post:
                raise _lib.B200Error(_lib.ERR_UNSUPPORTED, f"input_schedule({s.component!r}) must come before six_dof()")
        schedules = [s for s in pre if isinstance(s, InputSchedule)]
        self.pre_systems, self.post_systems = [s for s in pre if isinstance(s, HostSystem)], post
        # The reference's build yields an independent exec: this one owns private copies of the world's columns
        # (a later World.build() re-finalises the World's own buffers) and of the effector objects (the query-join
        # masks below are per build — the caller's effectors are never mutated).
        world = world._clone_for_exec()
        self.world = world
        self._effectors = [copy.copy(e) for e in self.six.effectors]
        for e in self._effectors:
            if isinstance(e, Effector):
                e.with_mask(None)
        self.n_worlds = int(n_worlds)
        self.sim_time_step = quantised_time_step(simulation_rate)
        self.ticks_per_telemetry = ticks_per_telemetry(simulation_rate, telemetry_rate)
        self.max_ticks = max_ticks
        world.finalize(self.n_worlds)
        # input schedules: cid -> (rows [T, n_worlds, n_owner, width], first_tick); the host keeps the rows for history
        self._schedules: Dict[int, tuple] = {}
        effector_cols = {component_id(e.column_name()) for e in self._effectors if e.column_name()}
        for s in schedules:
            cid = component_id(s.component)
            if cid in self._schedules:
                raise ValueError(f"two input_schedule()s drive column '{s.component}'")
            if cid not in effector_cols:
                raise ValueError(f"input_schedule({s.component!r}): not an input column of a six_dof() effector")
            if (world_params or {}).keys() & {s.component}:
                raise ValueError(f"world_params sets column '{s.component}', which an input_schedule drives")
            col = world.columns[cid]
            self._schedules[cid] = (_schedule_rows(s.component, s.rows, self.n_worlds, len(col.entity_ids), col.width),
                                    s.first_tick)
        for name, arr in (world_params or {}).items():
            col = world.columns[component_id(name)]
            col.buffer[...] = np.asarray(arr, dtype=col.dtype).reshape(col.buffer.shape)
        bodies = world.body_entities()
        # join rule (query.rs:672-710): every Body column must list the same entities in the same order
        for cname in ("world_vel", "world_accel", "force", "inertia"):
            col = world.columns.get(component_id(cname))
            if col is None or col.entity_ids != bodies:
                raise _lib.B200ValueError(_lib.ERR_COMPONENT_NOT_FOUND, f"component not found: {cname}")
        # Query join (query.rs:672-710): an effector only runs on the entities that own its input
        # component.  Full membership -> no mask; partial (order-preserving) membership -> entity mask +
        # a body-row-expanded copy of the column for the device; no members / foreign order -> error.
        self._partial: Dict[int, tuple] = {}
        for e in self._effectors:
            cname = e.column_name()
            if not cname:
                continue
            col = world.columns.get(component_id(cname))
            if col is None or not col.entity_ids:
                raise _lib.B200ValueError(_lib.ERR_COMPONENT_NOT_FOUND, f"component not found: {cname}")
            if col.entity_ids == bodies:
                continue
            rows = [bodies.index(ent) for ent in col.entity_ids if ent in bodies]
            if len(rows) != len(col.entity_ids) or rows != sorted(rows):
                raise _lib.B200ValueError(_lib.ERR_COMPONENT_NOT_FOUND, f"component not found: {cname} (owners are not Body entities)")
            mask = np.zeros(len(bodies), dtype=np.uint8)
            mask[rows] = 1
            e.with_mask(mask)
            self._partial[component_id(cname)] = (np.asarray(rows), np.zeros((self.n_worlds, len(bodies), col.width)))
        # Device-resident telemetry cycles (small interactive worlds): the state stays on the GPU for a whole
        # run() and every telemetry sample — all five Body columns — is recorded into the device trajectory
        # ring, read back in one transfer per `_ring_cap` cycles instead of one PCIe round trip per cycle.
        # Results are identical to the invoke_batch path (same kernels, same tick boundaries).
        n_bodies = len(bodies) * self.n_worlds
        if resident is None:
            resident = os.environ.get("B200_RESIDENT", "1") != "0" and 0 < n_bodies <= 65536
        self._ring_cap = 0
        if resident and n_bodies:
            ld = (n_bodies + 127) // 128 * 128
            self._ring_cap = int(max(1, min(4096, (64 << 20) // (25 * ld * 8))))
        # ticks of one invoke_batch stay in registers up to 32 at a time (no effect on results)
        self.backend = B200Exec(len(bodies), self.n_worlds, self.sim_time_step, self.six.time_step, self._effectors,
                                self.six.integrator.value, math, device, max_fused_ticks=32, world=world,
                                trajectory_every=self.ticks_per_telemetry if self._ring_cap else 0,
                                trajectory_capacity=self._ring_cap, trajectory_full=bool(self._ring_cap))
        for cid, (rows, first) in self._schedules.items():
            if cid in self._partial:  # body-row-expanded like the column the device holds
                full = np.zeros(rows.shape[:2] + (len(bodies), rows.shape[3]))
                full[:, :, self._partial[cid][0], :] = rows
                rows = full
            self.backend.set_schedule(cid, rows, first)
        self.tick = 0
        self.build_ms = 0.0
        self._prof = {"execute_buffers": [], "add_to_history": [], "h2d_upload": [], "kernel_invoke": [], "d2h_download": []}
        self.dirty: set = set()
        self._db = None
        self._history: Dict[int, List[np.ndarray]] = {cid: [] for cid in self.world.columns}
        self._globals_hist: List[tuple] = []
        self._record()

    # -- data plumbing -------------------------------------------------------------
    def _scheduled_value(self, cid: int, tick):
        """Host value of a scheduled column after the tick whose Tick value is `tick` (array: one per tick)."""
        rows, first = self._schedules[cid]
        return rows[schedule_row(tick, first, rows.shape[0])]

    def _record(self) -> None:
        for cid, col in self.world.columns.items():
            self._history[cid].append(col.buffer.copy())
        self._globals_hist.append((self.tick, self.sim_time_step))
        if getattr(self, "_db", None) is not None:
            self._db.flush()  # commit_world_head_unified: one row per (entity, component) per telemetry cycle

    def _bind_buffers(self) -> None:
        """Pointer tables for invoke_batch, built once: inputs are the world's own column buffers
        (updated in place, so the addresses are stable), outputs are executor-owned buffers that never
        alias an input (cranelift_exec.rs:101-107,138-154)."""
        be = self.backend
        self._tick_in = np.zeros(1, dtype=np.uint64)
        self._dt_in = np.array([self.sim_time_step])
        self._ins, self._outs = [], []
        for cid in be.input_ids:
            if cid == component_id("tick"):
                self._ins.append(self._tick_in)
            elif cid == component_id("simulation_time_step"):
                self._ins.append(self._dt_in)
            elif cid in self._schedules:
                self._ins.append(None)  # the device-resident schedule drives it
            elif cid in self._partial:
                self._ins.append(self._partial[cid][1])  # body-row-expanded copy, refreshed before every invoke
            else:
                buf = self.world.columns[cid].buffer
                assert buf.flags.c_contiguous and buf.nbytes == be.column_bytes(cid)
                self._ins.append(buf)
        for cid in be.output_ids:
            if cid in (component_id("tick"), component_id("simulation_time_step")):
                self._outs.append(np.zeros(1, dtype=np.uint64 if cid == component_id("tick") else np.float64))
            elif cid in self._schedules:
                self._outs.append(None)  # known on the host: the row of the last tick
            elif cid in self._partial:
                self._outs.append(np.empty_like(self._partial[cid][1]))
            else:
                self._outs.append(np.empty_like(self.world.columns[cid].buffer))
        self._in_ptrs = [None if a is None else a.ctypes.data for a in self._ins]
        self._out_ptrs = [None if a is None else a.ctypes.data for a in self._outs]

    def _invoke(self, n: int) -> None:
        """WorldExec::run -> invoke_batch (cranelift_exec.rs:284-303,129-195)."""
        be = self.backend
        if not hasattr(self, "_in_ptrs"):
            self._bind_buffers()
        self._tick_in[0] = self.tick
        self._dt_in[0] = self.sim_time_step
        for cid, (rows, expanded) in self._partial.items():
            if cid not in self._schedules:
                expanded[:, rows, :] = self.world.columns[cid].buffer
        be.invoke_batch_ptrs(self._in_ptrs, self._out_ptrs, n)
        for cid, buf in zip(be.output_ids, self._outs):
            if cid == component_id("tick"):
                self.tick = int(buf[0])  # world.advance_tick() x n
            elif cid != component_id("simulation_time_step") and cid not in self._partial and buf is not None:
                col = self.world.columns[cid]
                if col.buffer.nbytes != buf.nbytes:
                    raise _lib.B200ValueError(_lib.ERR_VALUE_SIZE_MISMATCH, "value size mismatch")
                np.copyto(col.buffer, buf)
        for cid in self._schedules:
            np.copyto(self.world.columns[cid].buffer, self._scheduled_value(cid, self.tick - 1))

    def _run_resident(self, cycles: int) -> None:
        """`cycles` whole telemetry cycles without leaving the device: upload the host columns once, step,
        read the recorded samples back per ring-full, leave the final state in the host columns."""
        be = self.backend
        tpt = self.ticks_per_telemetry
        tick_id, dt_id = component_id("tick"), component_id("simulation_time_step")
        t0 = time.perf_counter()
        for cid in be.input_ids:
            if cid == tick_id:
                be.upload(cid, np.array([self.tick], dtype=np.uint64))
            elif cid == dt_id:
                be.upload(cid, np.array([self.sim_time_step]))
            elif cid in self._schedules:
                continue  # the device-resident schedule drives it
            elif cid in self._partial:
                rows, expanded = self._partial[cid]
                expanded[:, rows, :] = self.world.columns[cid].buffer
                be.upload(cid, expanded)
            else:
                be.upload(cid, self.world.columns[cid].buffer)
        upload_ms = (time.perf_counter() - t0) * 1e3
        body_cols = [(component_id("world_pos"), 0, 7), (component_id("world_vel"), 7, 13),
                     (component_id("world_accel"), 13, 19), (component_id("force"), 19, 25)]
        sampled = {cid for cid, _, _ in body_cols}
        while cycles > 0:
            c = min(cycles, self._ring_cap)
            t0 = time.perf_counter()
            be.trajectory_reset()
            be.step(c * tpt)
            traj = be.trajectory()                                   # [c, n_worlds, n_bodies, 25]
            run_ms = (time.perf_counter() - t0) * 1e3 + upload_ms
            upload_ms = 0.0
            t_hist = time.perf_counter()
            for cid, lo, hi in body_cols:                            # one contiguous block per column, rows are views
                self._history[cid].extend(np.ascontiguousarray(traj[:, :, :, lo:hi]))
            last_ticks = self.tick + (np.arange(c) + 1) * tpt - 1         # Tick value of each cycle's last tick
            for cid, col in self.world.columns.items():
                if cid in self._schedules:                           # the row each cycle's last tick used
                    vals = self._scheduled_value(cid, last_ticks)
                    self._history[cid].extend(vals)
                    np.copyto(col.buffer, vals[-1])
                elif cid not in sampled:                             # not written by six_dof(): pass-through
                    self._history[cid].extend([col.buffer.copy()] * c)
            self._globals_hist.extend((self.tick + (k + 1) * tpt, self.sim_time_step) for k in range(c))
            self.tick += c * tpt
            for cid, lo, hi in body_cols:
                np.copyto(self.world.columns[cid].buffer, traj[-1, :, :, lo:hi])
            if getattr(self, "_db", None) is not None:
                self._db.flush()  # the c cycles of this ring read-back, each with its own timestamp
            hist_ms = (time.perf_counter() - t_hist) * 1e3
            self._prof["execute_buffers"] += [run_ms / c] * c
            self._prof["add_to_history"] += [hist_ms / c] * c
            for k_dst in ("h2d_upload", "kernel_invoke", "d2h_download"):
                self._prof[k_dst] += [0.0] * c                        # not separable on this path
            cycles -= c

    # -- public API ------------------------------------------------------------------
    def run(self, ticks: int = 1, show_progress: bool = True, is_canceled=None, pre_step=None, post_step=None):
        """exec.rs:111-173: `while remaining > 0 { exec.run(); commit_world_head }` — one
        invoke_batch of ticks_per_telemetry ticks per cycle, a history row per cycle.  Runs without host
        callbacks take the device-resident route for their whole cycles (same rows, one transfer)."""
        remaining = int(ticks)
        host_cb = bool(self.pre_systems or self.post_systems or pre_step or post_step)
        if self._ring_cap and not host_cb and is_canceled is None and remaining >= self.ticks_per_telemetry:
            whole = remaining // self.ticks_per_telemetry
            self._run_resident(whole)
            remaining -= whole * self.ticks_per_telemetry
        while remaining > 0:
            n = min(self.ticks_per_telemetry, remaining)
            per_call = 1 if host_cb else n
            done = 0
            while done < n:
                ctx = StepContext(self)
                if pre_step:
                    pre_step(self.tick, ctx)
                for s in self.pre_systems:
                    s.fn(ctx)
                t_inv = time.perf_counter()
                self._invoke(per_call)
                self._prof["execute_buffers"].append((time.perf_counter() - t_inv) * 1e3 * (n / per_call))
                tm = self.backend.timings()
                for k_src, k_dst in (("h2d_upload_ms", "h2d_upload"), ("kernel_invoke_ms", "kernel_invoke"), ("d2h_download_ms", "d2h_download")):
                    self._prof[k_dst].append(tm[k_src])
                for s in self.post_systems:
                    s.fn(ctx)
                if post_step:
                    post_step(self.tick, ctx)
                done += per_call
            t_hist = time.perf_counter()
            self._record()
            self._prof["add_to_history"].append((time.perf_counter() - t_hist) * 1e3)
            remaining -= n
            # like the reference (exec.rs:130-165): run the batch, commit it, then ask
            if is_canceled is not None and is_canceled():
                break
        return self

    def history(self, names: Union[str, Sequence[str]]):
        """`exec.history("e1.world_pos")` -> {name: rows[T, width]} (world 0; use
        `history_worlds` for the batch).  The reference returns a polars frame."""
        if isinstance(names, str):
            names = [names]
        out = {}
        for pair in names:
            ent, comp = pair.rsplit(".", 1)
            cid = component_id(comp)
            if ent.lower() == "globals":
                vals = [g[0] if comp == "tick" else g[1] for g in self._globals_hist]
                out[pair] = np.asarray(vals).view(_Series)
                continue
            col = self.world.columns.get(cid)
            if col is None:
                raise _lib.B200ValueError(_lib.ERR_COMPONENT_NOT_FOUND, f"component not found: {pair}")
            row = col.row_of(self.world.entity_by_name(ent))
            out[pair] = np.stack([h[0, row] for h in self._history[cid]]).view(_Series)
        return out

    def attach_db(self, path: str, start_timestamp_us: Optional[int] = None, world: int = 0):
        """Stream the telemetry of world `world` into an elodin-db directory while the run is in flight: `init_db` now
        (every pair registered, the rows recorded so far committed), then one commit per telemetry cycle
        (`commit_world_head_unified`, impeller2_server.rs:390-438) — per ring read-back on the device-resident route.
        `close_db()` finishes the directory."""
        from . import db_sink

        if getattr(self, "_db", None) is not None:
            raise _lib.B200Error(_lib.ERR_INVALID_ARGUMENT, "a database is already attached")
        self._db = (db_sink.LiveDbWriter(self, path, world=world) if start_timestamp_us is None
                    else db_sink.LiveDbWriter(self, path, start_timestamp_us, world))
        return self._db

    def close_db(self):
        db, self._db = getattr(self, "_db", None), None
        return db.close() if db is not None else None

    def write_db(self, path: str, start_timestamp_us: Optional[int] = None, world: int = 0):
        """Write the recorded telemetry as an elodin-db directory (`elodin_b200.db_sink`): what the
        reference's `init_db` + `commit_world_head_unified` leave on disk for `elodin-db export` / the editor."""
        from . import db_sink

        if start_timestamp_us is None:
            return db_sink.write_db(self, path, world=world)
        return db_sink.write_db(self, path, start_timestamp_us, world)

    def history_worlds(self, pair: str) -> np.ndarray:
        ent, comp = pair.rsplit(".", 1)
        col = self.world.columns[component_id(comp)]
        row = col.row_of(self.world.entity_by_name(ent))
        return np.stack([h[:, row] for h in self._history[col.component.id]])

    def column_array(self, cid) -> np.ndarray:
        cid = component_id(cid) if isinstance(cid, str) else int(cid)
        return self.world.columns[cid].buffer[0]

    def profile(self) -> dict:
        """Profiler::profile (libs/nox-py/src/profile.rs:28-56): mean ms per telemetry cycle and
        real_time_factor = time_step * ticks_per_telemetry / tick (history/DB commit included
        the way the reference includes add_to_history)."""
        mean = lambda k: float(np.mean(self._prof[k])) if self._prof[k] else 0.0
        tick = mean("execute_buffers") + mean("add_to_history")
        batch_ms = self.sim_time_step * 1e3 * max(self.ticks_per_telemetry, 1)
        out = {"build": self.build_ms, "copy_to_client": 0.0, "execute_buffers": mean("execute_buffers"), "copy_to_host": 0.0,
               "h2d_upload": mean("h2d_upload"), "kernel_invoke": mean("kernel_invoke"), "d2h_download": mean("d2h_download"),
               "add_to_history": mean("add_to_history"), "tick": tick, "time_step": self.sim_time_step * 1e3,
               "ticks_per_telemetry": float(self.ticks_per_telemetry),
               "real_time_factor": (batch_ms / tick) if tick > 0 else float("inf")}
        out.update({"backend": self.backend.timings()})
        return out
