"""Input schedules: effector input columns driven by per-tick rows held on the device.

Every GPU test checks the row rule of b200_sixdof_set_schedule — the tick whose Tick value is k reads row
clamp(k - first_tick, 0, T - 1) — against the CPU oracle stepped tick by tick with that row as the column, or against
the same run without a schedule.  The CPU tests cover the host side of el.input_schedule.
"""

import numpy as np
import pytest

import elodin_b200 as el
from elodin_b200 import _lib
from elodin_b200.executor import FORCE, INERTIA, WORLD_ACCEL, WORLD_POS, WORLD_VEL
from tests.util import random_world

FAST_TOL_TICK = 1e-12
DT = 1.0 / 120.0
T_ROWS, FIRST, N_TICKS = 7, 2, 12  # ticks 0..1 before the table, 2..8 inside it, 9..11 after it


def _state(ex):
    return [ex.download(c) for c in (WORLD_POS, WORLD_VEL, WORLD_ACCEL, FORCE)]


def _assert_exact(got, want, what=""):
    for name, a, b in zip(("pos", "vel", "accel", "force"), got, want):
        assert np.array_equal(a, b), f"{what} {name}: max abs diff {np.max(np.abs(a - b))}"


def _assert_close(got, want, tol, what=""):
    for name, a, b in zip(("pos", "vel", "accel", "force"), got, want):
        scale = max(np.max(np.abs(b)), 1e-300)
        err = float(np.max(np.abs(a - b)) / scale)
        assert err <= tol, f"{what} {name}: rel err {err:.3e} > {tol}"


# ----------------------------------------------------------------------------------------- effector lists

def _case(kind, M, N, seed=7):
    """(elodin effectors, oracle effector builder, plain columns, schedules) of one effector list.  The builder maps
    {column name: [M, N, width]} to the oracle list for one tick."""
    rng = np.random.default_rng(seed)
    if kind == "rocket":  # rocket/main.py: gravity + thrust + body wrench, thrust and wrench scheduled
        effs = [el.GravityConst((0.0, 0.0, -9.81)), el.ThrustBody((-1.0, 0.0, 0.0), "thrust"), el.WrenchBody("aero_force")]
        scheds = {"thrust": rng.uniform(0.0, 400.0, (T_ROWS, M, N, 1)), "aero_force": rng.normal(0.0, 5.0, (T_ROWS, M, N, 6))}

        def oracle_effs(O, c):
            return [O.Effector(O.EFF_GRAVITY_CONST, p=(0, 0, -9.81)), O.Effector(O.EFF_THRUST_BODY, p=(-1.0, 0, 0), column=c["thrust"]),
                    O.Effector(O.EFF_WRENCH_BODY, column=c["aero_force"])]
        return effs, oracle_effs, {}, scheds
    if kind == "ball":  # ball/sim.py: gravity + quadratic drag, the wind scheduled
        effs = [el.GravityConst((0.0, 0.0, -9.81)), el.DragQuadratic(0.6125, 0.25, "wind")]
        scheds = {"wind": rng.normal(0.0, 8.0, (T_ROWS, M, N, 3))}

        def oracle_effs(O, c):
            return [O.Effector(O.EFF_GRAVITY_CONST, p=(0, 0, -9.81)), O.Effector(O.EFF_DRAG_QUADRATIC, p=(0.6125, 0.25), column=c["wind"])]
        return effs, oracle_effs, {}, scheds
    raise KeyError(kind)


def _oracle(O, pos, vel, ine, oracle_effs, columns, n_ticks, integrator="rk4", tick0=0):
    """The oracle stepped tick by tick; `columns(k)` is {name: [M, N, width]} for the tick whose Tick value is k."""
    w = O.World(pos, vel, ine)
    for t in range(n_ticks):
        effs = oracle_effs(O, columns(tick0 + t))
        if integrator == "rk4":
            w.rk4(DT, 1, effs)
        else:
            w.semi_implicit(DT, 1, effs)
    return w.pos, w.vel, w.accel, w.force


def _rows_at(scheds, first=FIRST):
    return lambda k: {n: r[el.schedule_row(k, first, r.shape[0])] for n, r in scheds.items()}


def _run(M, N, effs, scheds, pos, vel, ine, math, integrator="rk4", fused=32, n_ticks=N_TICKS, first=FIRST, cols=None):
    with el.B200Exec(N, M, DT, None, effs, integrator, math, max_fused_ticks=fused) as ex:
        ex.set_state(pos, vel, ine, **(cols or {}))
        for name, rows in scheds.items():
            ex.set_schedule(name, rows, first)
        ex.step(n_ticks, sync=True)
        return _state(ex)


# ----------------------------------------------------------------------------------------- CPU: host side

def _motor_world(n_bodies=2, owners=None):
    Thrust = el.Annotated[np.ndarray, el.Component("thrust", el.ComponentType.F64)]

    @el.dataclass
    class Motor(el.Archetype):
        thrust: Thrust

    w = el.World()
    for i in range(n_bodies):
        arch = [el.Body()]
        if owners is None or i in owners:
            arch.append(Motor(np.array([0.0])))
        w.spawn(arch, name=f"b{i}")
    return w


def test_schedule_row_rule():
    """clamp(k - first_tick, 0, T - 1): the first row before the table, the last one after it."""
    ticks = np.arange(12)
    want = [0, 0, 0, 1, 2, 3, 4, 5, 6, 6, 6, 6]
    assert list(el.schedule_row(ticks, 2, 7)) == want
    assert int(el.schedule_row(0, 0, 1)) == 0 and int(el.schedule_row(10 ** 9, 0, 1)) == 0
    assert int(el.schedule_row(5, 10, 3)) == 0 and int(el.schedule_row(11, 10, 3)) == 1


def test_input_schedule_shapes_and_broadcast():
    from elodin_b200.world import _schedule_rows

    curve = np.arange(5.0)
    a = _schedule_rows("thrust", curve[:, None], 3, 1, 1)           # [T, n_owner] with width 1
    assert a.shape == (5, 3, 1, 1) and np.array_equal(a[:, 2, 0, 0], curve)
    b = _schedule_rows("wind", np.ones((4, 2, 3)), 3, 2, 3)         # [T, n_owner, width]: broadcast over worlds
    assert b.shape == (4, 3, 2, 3) and b.flags.c_contiguous
    c = np.random.default_rng(0).normal(size=(4, 3, 2, 3))
    assert np.array_equal(_schedule_rows("wind", c, 3, 2, 3), c)     # per world
    for bad in (np.ones((4, 2)), np.ones((4, 2, 2)), np.ones((4, 2, 2, 3)), np.ones((0, 2, 3)), np.ones(4)):
        with pytest.raises(ValueError, match="wind"):
            _schedule_rows("wind", bad, 3, 2, 3)
    s = el.input_schedule("thrust", curve[:, None], first_tick=3)
    assert isinstance(s, el.InputSchedule) and s.first_tick == 3 and s.component == "thrust"
    with pytest.raises(ValueError):
        el.input_schedule("thrust", curve[:, None], first_tick=-1)
    assert isinstance(el.input_schedule("thrust", curve[:, None]) | el.six_dof(), el.Pipe)


def _exec_without_backend(world, system, world_params=None, n_worlds=1):
    """Exec.__init__ up to (not including) the backend: the host checks run without a GPU."""
    class _Stop(Exception):
        pass

    import elodin_b200.world as W
    real = W.B200Exec

    def stop(*a, **k):
        raise _Stop()
    W.B200Exec = stop
    try:
        world.build(system, n_worlds=n_worlds, world_params=world_params)
    except _Stop:
        return True
    finally:
        W.B200Exec = real
    return False


def test_input_schedule_conflicts_are_errors():
    effs = el.GravityConst((0.0, 0.0, -9.81)) | el.ThrustBody((-1.0, 0.0, 0.0), "thrust")
    rows = np.ones((4, 2))
    w = _motor_world()
    # a valid program reaches the backend
    assert _exec_without_backend(w, el.input_schedule("thrust", rows) | el.six_dof(sys=effs))
    with pytest.raises(ValueError, match="thrust"):  # world_params would be overwritten every tick
        _exec_without_backend(w, el.input_schedule("thrust", rows) | el.six_dof(sys=effs), world_params={"thrust": np.ones((1, 2, 1))})
    with pytest.raises(ValueError, match="world_vel"):  # not an effector input column
        _exec_without_backend(w, el.input_schedule("world_vel", np.ones((4, 2, 6))) | el.six_dof(sys=effs))
    with pytest.raises(ValueError, match="thrust"):  # two schedules for one column
        _exec_without_backend(w, el.input_schedule("thrust", rows) | el.input_schedule("thrust", rows) | el.six_dof(sys=effs))
    with pytest.raises(ValueError, match="thrust"):  # wrong owner count
        _exec_without_backend(w, el.input_schedule("thrust", np.ones((4, 3))) | el.six_dof(sys=effs))
    with pytest.raises(_lib.B200Error):  # after six_dof()
        _exec_without_backend(w, el.six_dof(sys=effs) | el.input_schedule("thrust", rows))


def test_step_context_refuses_scheduled_columns():
    class _Exec:
        _schedules = {el.component_id("thrust"): (np.zeros((1, 1, 1, 1)), 0)}
        world = None
    ctx = el.StepContext(_Exec())
    with pytest.raises(ValueError, match="thrust"):
        ctx.column("thrust")
    with pytest.raises(ValueError, match="thrust"):
        ctx.write_component("b0.thrust", 1.0)


def test_history_of_a_scheduled_column_follows_the_row_rule():
    """The host-side history rows: the row of each cycle's last tick, in owner layout (partial membership kept)."""
    from elodin_b200.world import Exec

    ex = Exec.__new__(Exec)
    rows = np.arange(7.0).reshape(7, 1, 1, 1) * np.array([1.0, 10.0]).reshape(1, 1, 2, 1)
    ex._schedules = {1: (rows, 2)}
    got = ex._scheduled_value(1, np.array([0, 1, 2, 5, 8, 9, 40]))
    assert got.shape == (7, 1, 2, 1)
    assert list(got[:, 0, 0, 0]) == [0.0, 0.0, 0.0, 3.0, 6.0, 6.0, 6.0]
    assert list(got[:, 0, 1, 0]) == [0.0, 0.0, 0.0, 30.0, 60.0, 60.0, 60.0]


# ----------------------------------------------------------------------------------------- GPU

gpu = pytest.mark.gpu
CASES = [(kind, M, N) for kind in ("rocket", "ball") for (M, N) in ((1, 1), (3, 5), (64, 7))]


@gpu
@pytest.mark.parametrize("kind,M,N", CASES)
def test_exact_fused_schedule_matches_oracle(oracle, kind, M, N):
    """12 ticks in ONE step call (max_fused_ticks = 32) across the table's start and end: bit-identical to the
    oracle stepped tick by tick with the row of each tick."""
    pos, vel, ine = random_world(11, M, N)
    effs, oeffs, cols, scheds = _case(kind, M, N)
    got = _run(M, N, effs, scheds, pos, vel, ine, "exact")
    want = _oracle(oracle, pos, vel, ine, oeffs, _rows_at(scheds), N_TICKS)
    _assert_exact(got, want, f"{kind} M={M} N={N}")


@gpu
@pytest.mark.parametrize("integrator", ["rk4", "semi_implicit"])
@pytest.mark.parametrize("route", ["spec", "interpreter"])
@pytest.mark.parametrize("kind,M,N", CASES)
def test_fast_fused_schedule_matches_oracle(oracle, kind, M, N, route, integrator):
    """The same in FAST arithmetic, within 12 x FAST_TOL_TICK: the specialised kernel, and the interpreter kernel (an
    all-true entity mask takes every list off the signatures)."""
    pos, vel, ine = random_world(12, M, N)
    effs, oeffs, cols, scheds = _case(kind, M, N)
    if route == "interpreter":
        effs = [e.with_mask(np.ones(N, dtype=np.uint8)) for e in effs]
    got = _run(M, N, effs, scheds, pos, vel, ine, "fast", integrator)
    want = _oracle(oracle, pos, vel, ine, oeffs, _rows_at(scheds), N_TICKS, integrator)
    _assert_close(got, want, N_TICKS * FAST_TOL_TICK, f"{kind} {route} {integrator} M={M} N={N}")


@gpu
@pytest.mark.parametrize("math", ["fast", "exact"])
def test_body_pair_kernel_with_a_per_world_thrust_schedule(oracle, math):
    """2^17 + 1 worlds (the body-pair kernel, with an odd tail), the rocket set, fused ticks, a thrust schedule that
    differs per world; a strided sample of worlds against the oracle."""
    M, N = (1 << 17) + 1, 1
    rng = np.random.default_rng(3)
    pos = np.tile(np.array([0, 0, 0, 1.0, 0, 0, 10.0]), (M, 1, 1))
    q = rng.normal(size=(M, 1, 4))
    pos[..., :4] = q / np.linalg.norm(q, axis=-1, keepdims=True)
    vel = np.concatenate([rng.normal(0, 0.1, (M, 1, 3)), rng.normal(0, 5, (M, 1, 3))], -1)
    ine = np.tile(np.array([0.1, 1.0, 1.0, 0, 0, 0, 3.0]), (M, 1, 1))
    wind = rng.normal(0, 3, (M, 1, 3))
    thrust = rng.uniform(0, 300, (T_ROWS, M, 1, 1))
    effs = [el.GravityConst((0.0, 0.0, -9.81)), el.ThrustBody((-1.0, 0.0, 0.0), "thrust"), el.DragQuadratic(0.6125, 0.0025, "wind")]
    got = _run(M, N, effs, {"thrust": thrust}, pos, vel, ine, math, fused=100, cols={"wind": wind})
    idx = np.r_[np.arange(0, M, 1021), M - 2, M - 1]
    sub = lambda a: np.ascontiguousarray(a[idx])

    def oeffs(O, c):
        return [O.Effector(O.EFF_GRAVITY_CONST, p=(0, 0, -9.81)), O.Effector(O.EFF_THRUST_BODY, p=(-1.0, 0, 0), column=c["thrust"]),
                O.Effector(O.EFF_DRAG_QUADRATIC, p=(0.6125, 0.0025), column=sub(wind))]
    want = _oracle(oracle, sub(pos), sub(vel), sub(ine), oeffs, _rows_at({"thrust": thrust[:, idx]}), N_TICKS)
    if math == "exact":
        _assert_exact([a[idx] for a in got], want, "body pair exact")
    else:
        _assert_close([a[idx] for a in got], want, N_TICKS * FAST_TOL_TICK, "body pair fast")


@gpu
@pytest.mark.parametrize("kind", ["rocket", "ball"])
def test_constant_rows_change_nothing(kind, record_property):
    """A schedule whose every row equals the column gives the unscheduled result: bit for bit in EXACT (fused and one
    tick per launch) and in FAST one-tick launches; FAST fused launches within tolerance (whether the bits match is
    recorded)."""
    M, N = 9, 4
    pos, vel, ine = random_world(21, M, N)
    effs, _, _, scheds = _case(kind, M, N)
    cols = {n: r[3] for n, r in scheds.items()}
    const = {n: np.broadcast_to(c, (T_ROWS,) + c.shape).copy() for n, c in cols.items()}
    for math, fused in (("exact", 32), ("exact", 1), ("fast", 1), ("fast", 32)):
        plain = _run(M, N, effs, {}, pos, vel, ine, math, fused=fused, cols=cols)
        sched = _run(M, N, effs, const, pos, vel, ine, math, fused=fused, cols=cols)
        if math == "fast" and fused > 1:
            _assert_close(sched, plain, N_TICKS * FAST_TOL_TICK, f"{kind} fast fused")
            same = all(np.array_equal(a, b) for a, b in zip(sched, plain))
            record_property(f"{kind}_fast_fused_bit_identical", same)
            print(f"{kind}: FAST fused constant-row schedule bit-identical to the plain column: {same}")
        else:
            _assert_exact(sched, plain, f"{kind} {math} fused={fused}")


def _invoke_inputs(ex, tick, arrays=None):
    ins = []
    for cid in ex.input_ids:
        if cid == el.component_id("tick"):
            ins.append(np.array([tick], dtype=np.uint64))
        elif cid == el.component_id("simulation_time_step"):
            ins.append(np.array([DT]))
        else:
            ins.append((arrays or {}).get(cid))
    return ins


@gpu
@pytest.mark.parametrize("math", ["exact", "fast"])
def test_rows_follow_the_tick_column(math):
    """The rows follow the Tick value: a trajectory reset between two step calls does not shift them; invoke_batch
    calls that carry the tick forward, and a first_tick offset folded into the table, give the rows of one long
    step."""
    M, N = 5, 3
    pos, vel, ine = random_world(31, M, N)
    effs, _, _, scheds = _case("rocket", M, N)
    ref = _run(M, N, effs, scheds, pos, vel, ine, math)
    with el.B200Exec(N, M, DT, None, effs, "rk4", math, max_fused_ticks=32) as ex:
        ex.set_state(pos, vel, ine)
        for n, r in scheds.items():
            ex.set_schedule(n, r, FIRST)
        ex.step(5)
        ex.trajectory_reset()
        ex.step(7, sync=True)
        assert ex.tick == N_TICKS
        _assert_exact(_state(ex), ref, "trajectory reset")
    with el.B200Exec(N, M, DT, None, effs, "rk4", math, max_fused_ticks=32) as ex:
        ex.set_state(pos, vel, ine)
        for n, r in scheds.items():
            ex.set_schedule(n, r, FIRST)
        for k0, n in ((0, 4), (4, 1), (5, 7)):
            outs = dict(zip(ex.output_ids, ex.invoke_batch(_invoke_inputs(ex, k0), n)))
            assert int(outs[el.component_id("tick")][0]) == k0 + n
        _assert_exact([outs[c] for c in (WORLD_POS, WORLD_VEL, WORLD_ACCEL, FORCE)], ref, "invoke_batch tick")
    # first_tick = 0 with the rows of ticks 0..11 spelled out, then held
    k = np.arange(N_TICKS + 3)
    flat = {n: r[el.schedule_row(k, FIRST, T_ROWS)] for n, r in scheds.items()}
    _assert_exact(_run(M, N, effs, flat, pos, vel, ine, math, first=0), ref, "first_tick offset")
    # a run that starts at Tick 4 reads from row 2
    with el.B200Exec(N, M, DT, None, effs, "rk4", math, max_fused_ticks=32) as ex:
        ex.set_state(pos, vel, ine)
        for n, r in scheds.items():
            ex.set_schedule(n, r[2:], FIRST + 2)
        ex.upload("tick", np.array([4], dtype=np.uint64))
        ex.step(N_TICKS, sync=True)
        shifted = _state(ex)
    _assert_exact(shifted, _run(M, N, effs, {n: r[2:] for n, r in scheds.items()}, pos, vel, ine, math, first=0), "start at tick 4")


@gpu
@pytest.mark.parametrize("math", ["exact", "fast"])
def test_pipelined_invoke_batch_equals_step(math):
    """World ranges of the pipelined invoke_batch (>= 1024 bodies, small chunks) read the same rows as one step."""
    M, N = 256, 5
    pos, vel, ine = random_world(41, M, N)
    effs, _, _, scheds = _case("rocket", M, N)
    ref = _run(M, N, effs, scheds, pos, vel, ine, math)
    with el.B200Exec(N, M, DT, None, effs, "rk4", math, max_fused_ticks=32, invoke_chunk_bodies=256) as ex:
        for n, r in scheds.items():
            ex.set_schedule(n, r, FIRST)
        state = {WORLD_POS: pos, WORLD_VEL: vel, INERTIA: ine, WORLD_ACCEL: np.zeros((M, N, 6)), FORCE: np.zeros((M, N, 6))}
        outs = dict(zip(ex.output_ids, ex.invoke_batch(_invoke_inputs(ex, 0, state), N_TICKS)))
        got = [outs[c] for c in (WORLD_POS, WORLD_VEL, WORLD_ACCEL, FORCE)]
        assert np.array_equal(outs[el.component_id("thrust")], scheds["thrust"][-1])  # the last tick's row
    if math == "exact":
        _assert_exact(got, ref, "pipelined")
    else:
        _assert_close(got, ref, 2 * FAST_TOL_TICK, "pipelined")


@gpu
def test_column_contract(oracle):
    M, N = 2, 3
    pos, vel, ine = random_world(51, M, N)
    effs, oeffs, _, scheds = _case("rocket", M, N)
    with el.B200Exec(N, M, DT, None, effs, "rk4", "exact", max_fused_ticks=32) as ex:
        ex.set_state(pos, vel, ine)
        plain_thrust = np.full((M, N, 1), 123.0)
        ex.upload("thrust", plain_thrust)
        ex.upload("aero_force", np.zeros((M, N, 6)))
        for n, r in scheds.items():
            ex.set_schedule(n, r, FIRST)
        assert np.array_equal(ex.download("thrust"), plain_thrust)  # no tick yet: the column is untouched
        ex.step(3)
        assert np.array_equal(ex.download("thrust"), scheds["thrust"][0])  # last tick 2 -> row 0
        ex.step(6)
        assert np.array_equal(ex.download("thrust"), scheds["thrust"][6])  # last tick 8 -> row 6
        # the schedule owns the column's input
        with pytest.raises(_lib.B200Error) as e:
            ex.invoke_batch(_invoke_inputs(ex, ex.tick, {el.component_id("thrust"): plain_thrust}), 1)
        assert e.value.code == _lib.ERR_INVALID_ARGUMENT and f"{el.component_id('thrust'):016x}" in str(e.value)
        with pytest.raises(_lib.B200Error) as e:
            ex.upload("thrust", plain_thrust)
        assert e.value.code == _lib.ERR_INVALID_ARGUMENT
        for rows, cid, code in ((np.ones((T_ROWS, M, N, 2)), "thrust", _lib.ERR_VALUE_SIZE_MISMATCH),
                                (np.ones((T_ROWS, M, N, 1)), "no_such_column", _lib.ERR_COMPONENT_NOT_FOUND),
                                (np.ones((T_ROWS, M, N, 6)), "world_vel", _lib.ERR_INVALID_ARGUMENT),
                                (np.ones((1, 1, 1, 1)), "tick", _lib.ERR_INVALID_ARGUMENT)):
            with pytest.raises(_lib.B200Error) as e:
                ex.set_schedule(cid, rows)
            assert e.value.code == code, (cid, e.value)
        # clear: the column keeps its last-used row, later ticks read the column again (uploads allowed again)
        ex.clear_schedule("thrust")
        assert np.array_equal(ex.download("thrust"), scheds["thrust"][6])
        ex.upload("thrust", plain_thrust)
        ex.step(3, sync=True)
        got = _state(ex)
        assert ex.tick == 12
    cols = lambda k: {"thrust": scheds["thrust"][el.schedule_row(k, FIRST, T_ROWS)] if k < 9 else plain_thrust,
                      "aero_force": scheds["aero_force"][el.schedule_row(k, FIRST, T_ROWS)]}
    _assert_exact(got, _oracle(oracle, pos, vel, ine, oeffs, cols, 12), "clear_schedule")
    # graph worlds do not take schedules
    edges = np.array([[0, 1], [1, 0]])
    geffs = [el.GravityEdges("newton", G=6.6743e-11, edges=edges), el.ThrustBody((-1.0, 0.0, 0.0), "thrust")]
    with el.B200Exec(2, 1, DT, None, geffs, "rk4", "exact") as ex:
        with pytest.raises(_lib.B200Error) as e:
            ex.set_schedule("thrust", np.ones((3, 1, 2, 1)))
        assert e.value.code == _lib.ERR_UNSUPPORTED and "graph" in str(e.value)


@gpu
def test_ecs_input_schedule_equals_host_system(oracle):
    """test_host_system_feeds_per_tick_inputs with el.input_schedule in place of the host system: the same history rows
    bit for bit, on the device-resident route (far fewer launches than ticks)."""
    Thrust = el.Annotated[np.ndarray, el.Component("thrust", el.ComponentType.F64)]

    @el.dataclass
    class Motor(el.Archetype):
        thrust: Thrust

    def world():
        w = el.World()
        q = el.Quaternion.from_euler([0.0, np.radians(70.0), 0.0])
        w.spawn([el.Body(world_pos=el.SpatialTransform(angular=q, linear=np.array([0.0, 0.0, 1.0])),
                         inertia=el.SpatialInertia(3.0, np.array([0.1, 1.0, 1.0]))), Motor(np.array([0.0]))], name="rocket")
        return w
    curve = lambda tick: 300.0 * np.exp(-0.05 * tick)

    @el.host_system
    def thrust(ctx):
        ctx.column("thrust")[...] = curve(ctx.tick)

    effectors = el.GravityConst((0.0, 0.0, -9.81)) | el.ThrustBody((-1.0, 0.0, 0.0), "thrust")
    host = world().build(thrust | el.six_dof(sys=effectors, integrator=el.Integrator.Rk4), simulation_rate=120.0)
    host.run(25)
    table = np.array([[curve(k)] for k in range(25)])
    sched = world().build(el.input_schedule("thrust", table) | el.six_dof(sys=effectors), simulation_rate=120.0)
    l0 = sched.backend.timings()["kernel_launches"]
    sched.run(25)
    launches = sched.backend.timings()["kernel_launches"] - l0
    pairs = [f"rocket.{c}" for c in ("world_pos", "world_vel", "world_accel", "force", "inertia", "thrust")] + ["Globals.tick"]
    hh, hs = host.history(pairs), sched.history(pairs)
    for p in pairs:
        assert hh[p].shape == hs[p].shape and np.array_equal(np.asarray(hh[p]), np.asarray(hs[p])), p
    assert hs["rocket.thrust"][-1][0] == curve(24) and int(hs["Globals.tick"][-1]) == 25
    assert launches < 25 // 2, launches


@gpu
def test_rocket_golden_replayed_in_one_step(golden, oracle, record_property):
    """The reference's rocket telemetry integrated for 100 ticks in ONE EXACT step from row 0, the recorded thrust and
    aero_force rows 1..100 as schedules: bit-identical to the oracle stepped tick by tick, and inside the reference's
    own gate (math.isclose, rel = abs = 1e-4) of every recorded row (the trajectory ring samples each tick)."""
    g = golden
    dt = float(g["rocket.simulation_time_step"][0, 0])
    effs = [el.GravityConst((0.0, 0.0, -9.81)), el.ThrustBody((-1.0, 0.0, 0.0), "thrust"), el.WrenchBody("aero_force")]
    thrust = g["rocket.thrust"][1:101].reshape(100, 1, 1, 1)
    aero = g["rocket.aero_force"][1:101].reshape(100, 1, 1, 6)
    p0, v0, i0, a0 = (g[f"rocket.{c}"][0][None, None] for c in ("world_pos", "world_vel", "inertia", "world_accel"))
    with el.B200Exec(1, 1, dt, None, effs, "rk4", "exact", max_fused_ticks=100, trajectory_every=1, trajectory_capacity=100,
                     trajectory_full=True) as ex:
        ex.set_state(p0, v0, i0, accel=a0)
        ex.set_schedule("thrust", thrust)
        ex.set_schedule("aero_force", aero)
        l0 = ex.timings()["kernel_launches"]
        ex.step(100, sync=True)
        assert ex.timings()["kernel_launches"] - l0 == 1
        got = _state(ex)
        traj = ex.trajectory()[:, 0, 0]  # [100, 25]: pos, vel, accel, force after ticks 1..100
    O = oracle
    w = O.World(p0, v0, i0, a0)
    for t in range(100):
        w.rk4(dt, 1, [O.Effector(O.EFF_GRAVITY_CONST, p=(0, 0, -9.81)), O.Effector(O.EFF_THRUST_BODY, p=(-1.0, 0, 0), column=thrust[t]),
                      O.Effector(O.EFF_WRENCH_BODY, column=aero[t])])
    _assert_exact(got, (w.pos, w.vel, w.accel, w.force), "rocket replay")
    worst = 0.0
    for name, lo, hi in (("world_pos", 0, 7), ("world_vel", 7, 13), ("world_accel", 13, 19), ("force", 19, 25)):
        a, ref = traj[:, lo:hi], g[f"rocket.{name}"][1:101]
        dev = np.abs(a - ref)
        assert np.all(dev <= np.maximum(1e-4 * np.maximum(np.abs(a), np.abs(ref)), 1e-4)), name
        worst = max(worst, float(np.max(dev)))
    assert np.array_equal(traj[-1, :7], got[0][0, 0]) and np.array_equal(traj[-1, 19:], got[3][0, 0])
    record_property("rocket_replay_max_abs_dev", worst)
    print(f"rocket replay, 100 ticks in one step: max |dev| from the recorded telemetry over rows 1..100 = {worst:.3e}")
