"""elodin_b200 — B200-native drop-in for the six_dof() hot path of elodin-sys/elodin.

The package mirrors the slice of the nox-py ECS surface that path needs (World,
Body, WorldPos/WorldVel/Force/Inertia columns, six_dof(), World.build()/run(),
Exec.run()/history()) and routes every tick through libb200_sixdof.so — hand-written
sm_100a CUDA kernels behind the C ABI in include/b200_sixdof.h.  There is no CPU
implementation here: importing works anywhere, but building an executor without
the CUDA library or without a GPU raises.

    import elodin_b200 as el
    w = el.World()
    w.spawn(el.Body(world_vel=el.SpatialMotion(linear=[1.0, 0, 0])), name="e1")
    exec = w.build(el.six_dof(1.0 / 60.0))
    exec.run()
    exec.history("e1.world_pos")
"""

from . import _lib, effectors
from ._lib import B200Error, B200ValueError, component_id
from .effectors import (DragQuadratic, GravityConst, GravityEGM08, GravityEdges, GravityFrame, GravityJ2, Pipe, System, ThrustBody,
                        TorqueBodyFold, WrenchBody, WrenchWorld, all_pairs_edges)
from .executor import B200Exec, device_count, pinned_empty, pinned_free
from .world import (Annotated, Archetype, Body, Component, ComponentType, Edge, EntityId, Exec, Force, HostSystem,
                    Inertia, InputSchedule, Integrator, PrimitiveType, Quaternion, Seed, SimulationTick, SimulationTimeStep,
                    SpatialForce, SpatialInertia, SpatialMotion, SpatialTransform, StepContext, World, WorldAccel,
                    WorldPos, WorldVel, dataclass, host_system, input_schedule, quantised_time_step, schedule_row, six_dof,
                    ticks_per_telemetry)

__all__ = [n for n in dir() if not n.startswith("_")]
