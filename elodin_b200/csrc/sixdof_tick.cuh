// Per-body tick functions of the six_dof() hot path, shared by every kernel that integrates bodies
// (body_kernels.cu, graph_kernels.cu: nbody_tick_fused_kernel / small_world_kernel).
//
//   exact_tick   one tick in EXACT arithmetic (literal operation order, bit-identical to the oracle)
//   fast_ticks   n ticks in FAST arithmetic, state in registers; templated on an effector
//                signature SIG: SIG_GENERIC interprets the effector list at run time, any other value
//                is a compile-time set of built-in effectors (SURVEY §2.4 K2) whose per-body inputs
//                arrive in registers (EffIn) — no interpreter loop, no dead members, no parameter reads.
#pragma once
#include "sixdof_device.cuh"
#include "sixdof_internal.h"

namespace b200 {

// ------------------------------------------------------------------ column access
__device__ __forceinline__ double ldp(const double *base, uint64_t ld, int plane, uint64_t b)
{
    return base[(uint64_t)plane * ld + b];
}
__device__ __forceinline__ void stp(double *base, uint64_t ld, int plane, uint64_t b, double v)
{
    base[(uint64_t)plane * ld + b] = v;
}

__device__ __forceinline__ Pose load_pose(const double *p, uint64_t ld, uint64_t b)
{
    Pose o;
    o.q = Quat{ldp(p, ld, 0, b), ldp(p, ld, 1, b), ldp(p, ld, 2, b), ldp(p, ld, 3, b)};
    o.x = Vec3{ldp(p, ld, 4, b), ldp(p, ld, 5, b), ldp(p, ld, 6, b)};
    return o;
}
__device__ __forceinline__ Motion load_motion(const double *p, uint64_t ld, uint64_t b)
{
    Motion m;
    m.ang = Vec3{ldp(p, ld, 0, b), ldp(p, ld, 1, b), ldp(p, ld, 2, b)};
    m.lin = Vec3{ldp(p, ld, 3, b), ldp(p, ld, 4, b), ldp(p, ld, 5, b)};
    return m;
}
__device__ __forceinline__ Inertia load_inertia(const double *p, uint64_t ld, uint64_t b)
{
    Inertia I;
    I.diag = Vec3{ldp(p, ld, 0, b), ldp(p, ld, 1, b), ldp(p, ld, 2, b)};
    I.m = ldp(p, ld, 6, b);
    return I;
}
__device__ __forceinline__ void store_pose(double *p, uint64_t ld, uint64_t b, const Pose &o)
{
    stp(p, ld, 0, b, o.q.i); stp(p, ld, 1, b, o.q.j); stp(p, ld, 2, b, o.q.k); stp(p, ld, 3, b, o.q.w);
    stp(p, ld, 4, b, o.x.x); stp(p, ld, 5, b, o.x.y); stp(p, ld, 6, b, o.x.z);
}
__device__ __forceinline__ void store_motion(double *p, uint64_t ld, uint64_t b, const Motion &m)
{
    stp(p, ld, 0, b, m.ang.x); stp(p, ld, 1, b, m.ang.y); stp(p, ld, 2, b, m.ang.z);
    stp(p, ld, 3, b, m.lin.x); stp(p, ld, 4, b, m.lin.y); stp(p, ld, 5, b, m.lin.z);
}

// slot of the telemetry sample due after `tick_after` ticks, if any
__device__ __forceinline__ bool traj_due(const StepParams &P, uint64_t tick_after, uint64_t &slot)
{
    if (P.traj_every == 0 || (tick_after % P.traj_every) != 0) return false;
    slot = tick_after / P.traj_every - 1;
    return slot < P.traj_capacity;
}
// Trajectory samples are written once and never read back by a kernel: streaming stores (evict-first) keep them from
// pushing the state planes out of the L2 the next launch starts from.
__device__ __forceinline__ void stp_stream(double *base, uint64_t ld, int plane, uint64_t b, double v)
{
    __stcs(base + (uint64_t)plane * ld + b, v);
}
__device__ __forceinline__ void traj_store_state(const StepParams &P, uint64_t b, uint64_t slot, const Pose &x, const Motion &v)
{
    double *t = P.traj + slot * (uint64_t)P.traj_planes * P.ld;
    stp_stream(t, P.ld, 0, b, x.q.i); stp_stream(t, P.ld, 1, b, x.q.j); stp_stream(t, P.ld, 2, b, x.q.k); stp_stream(t, P.ld, 3, b, x.q.w);
    stp_stream(t, P.ld, 4, b, x.x.x); stp_stream(t, P.ld, 5, b, x.x.y); stp_stream(t, P.ld, 6, b, x.x.z);
    stp_stream(t, P.ld, 7, b, v.ang.x); stp_stream(t, P.ld, 8, b, v.ang.y); stp_stream(t, P.ld, 9, b, v.ang.z);
    stp_stream(t, P.ld, 10, b, v.lin.x); stp_stream(t, P.ld, 11, b, v.lin.y); stp_stream(t, P.ld, 12, b, v.lin.z);
}
// B200_TRAJ_FULL: WorldAccel and Force as the tick leaves them in the ECS columns
__device__ __forceinline__ void traj_store_af(const StepParams &P, uint64_t b, uint64_t slot, const Motion &a, const Motion &f)
{
    double *t = P.traj + (slot * (uint64_t)P.traj_planes + 13ull) * P.ld;
    stp_stream(t, P.ld, 0, b, a.ang.x); stp_stream(t, P.ld, 1, b, a.ang.y); stp_stream(t, P.ld, 2, b, a.ang.z);
    stp_stream(t, P.ld, 3, b, a.lin.x); stp_stream(t, P.ld, 4, b, a.lin.y); stp_stream(t, P.ld, 5, b, a.lin.z);
    stp_stream(t, P.ld, 6, b, f.ang.x); stp_stream(t, P.ld, 7, b, f.ang.y); stp_stream(t, P.ld, 8, b, f.ang.z);
    stp_stream(t, P.ld, 9, b, f.lin.x); stp_stream(t, P.ld, 10, b, f.lin.y); stp_stream(t, P.ld, 11, b, f.lin.z);
}

// ================================================================== EXACT body kernel

// edge_fold gravity of one body at the three stage positions, held in registers by the kernels that
// compute it themselves (small_world_kernel) instead of reading the gforce planes
struct GravReg {
    Vec3 g0, g1, g2;
    bool has; // the body owns >= 1 out-edge
};
__device__ __forceinline__ Vec3 grav_slot(const GravReg &g, int slot) { return slot == 0 ? g.g0 : (slot == 1 ? g.g1 : g.g2); }

// python/elodin/j2.py:5-29 in the operation order of oracle/sixdof_oracle.c:eff_gravity_j2.  Out of line: its pow()
// (the reference's `norm**6.0` is a float-exponent lax.pow) would otherwise cost every EXACT kernel registers.
static __device__ __noinline__ Vec3 j2_field_exact(double mu, double J2, double r_ref, Vec3 r, double m)
{
    using namespace ex;
    const double norm = sqr(dot3(r));
    const Vec3 e_r = div3(r, norm);
    const double n3 = mul(mul(norm, norm), norm);
    const double c0 = mul(-mu, m);
    const double n2 = mul(norm, norm), n4 = mul(n2, n2), n5 = mul(norm, n4);
    const double n6 = pow(norm, 6.0);
    const double kz = div(mul(3.0, r.z), n5);
    const double kr = sub(div(3.0, mul(2.0, n4)), div(mul(15.0, mul(r.z, r.z)), mul(2.0, n6)));
    const double c1 = mul(mul(c0, J2), mul(r_ref, r_ref));
    const Vec3 pm = div3(Vec3{mul(c0, r.x), mul(c0, r.y), mul(c0, r.z)}, n3); // the point-mass term
    return Vec3{add(pm.x, mul(c1, add(mul(kz, 0.0), mul(kr, e_r.x)))),
                add(pm.y, mul(c1, add(mul(kz, 0.0), mul(kr, e_r.y)))),
                add(pm.z, mul(c1, add(mul(kz, 1.0), mul(kr, e_r.z))))};
}

// clear_forces | effectors (array order) on the stage state; six_dof.rs:148-150,195
// One effector applied to the accumulating Force of a stage, in EXACT arithmetic.  `kind` is E.kind for the run-time
// interpreter and a compile-time constant for effector sequences (the switch then folds away).
// SCHED: the launch carries input schedules; the effector's column is the row of `tick` (the tick being integrated)
template <bool GREG, bool SCHED = false>
__device__ __forceinline__ void apply_effector_exact(uint32_t kind, const EffDev &E, const StepParams &P, uint64_t b, int slot,
                                                     const Pose &sx, const ex::PoseInv &pi, const Motion &sv, const Inertia &I,
                                                     const GravReg &greg, Motion &F, uint64_t tick = 0)
{
    using namespace ex;
    // the column base at each use (unscheduled launches read E.col there, exactly as without schedules)
    auto col = [&]() { return SCHED ? schedule_ptr(E.col, E.sched, tick) : E.col; };
    switch (kind) {
    case B200_EFF_GRAVITY_CONST: { // ball/sim.py:56-58: f + SpatialForce(linear=g*m)
        F.ang = Vec3{add(F.ang.x, 0.0), add(F.ang.y, 0.0), add(F.ang.z, 0.0)};
        F.lin = Vec3{add(F.lin.x, mul(E.p[0], I.m)), add(F.lin.y, mul(E.p[1], I.m)),
                     add(F.lin.z, mul(E.p[2], I.m))};
        break;
    }
    case B200_EFF_DRAG_QUADRATIC: { // ball/sim.py:99-116; result torque is zero
        double w0 = 0.0, w1 = 0.0, w2 = 0.0;
        if (col()) { w0 = ldp(col(), P.ld, 0, b); w1 = ldp(col(), P.ld, 1, b); w2 = ldp(col(), P.ld, 2, b); }
        const Vec3 fl = {sub(w0, sv.lin.x), sub(w1, sv.lin.y), sub(w2, sv.lin.z)};
        const double speed = sqr(dot3(fl));
        const double cd_rho = E.col_width == 5 ? ldp(col(), P.ld, 3, b) : E.p[0];
        const double area = E.col_width == 5 ? ldp(col(), P.ld, 4, b) : E.p[1];
        const double drag = mul(0.5, mul(mul(cd_rho, mul(speed, speed)), area));
        const Vec3 dir = div3(fl, speed);
        F.ang = Vec3{0.0, 0.0, 0.0};
        F.lin = Vec3{add(F.lin.x, mul(drag, dir.x)), add(F.lin.y, mul(drag, dir.y)), add(F.lin.z, mul(drag, dir.z))};
        break;
    }
    case B200_EFF_THRUST_BODY: { // rocket/main.py:429-431
        const double t = col() ? ldp(col(), P.ld, 0, b) : 0.0;
        const Vec3 d = qrot_with(sx.q, pi.qi, Vec3{E.p[0], E.p[1], E.p[2]});
        F.ang = Vec3{add(F.ang.x, 0.0), add(F.ang.y, 0.0), add(F.ang.z, 0.0)};
        F.lin = Vec3{add(F.lin.x, mul(d.x, t)), add(F.lin.y, mul(d.y, t)), add(F.lin.z, mul(d.z, t))};
        break;
    }
    case B200_EFF_WRENCH_BODY: { // rocket/main.py:407-413, falcon9/sim.py:659-672
        Vec3 a = {0.0, 0.0, 0.0}, c = {0.0, 0.0, 0.0};
        if (col()) {
            a = Vec3{ldp(col(), P.ld, 0, b), ldp(col(), P.ld, 1, b), ldp(col(), P.ld, 2, b)};
            c = Vec3{ldp(col(), P.ld, 3, b), ldp(col(), P.ld, 4, b), ldp(col(), P.ld, 5, b)};
        }
        const bool lin_first = (E.flags & B200_EFF_FLAG_WRENCH_LINEAR_FIRST) != 0;
        const Vec3 tw = qrot_with(sx.q, pi.qi, lin_first ? c : a);
        const Vec3 fw = qrot_with(sx.q, pi.qi, lin_first ? a : c);
        F.ang = Vec3{add(F.ang.x, tw.x), add(F.ang.y, tw.y), add(F.ang.z, tw.z)};
        F.lin = Vec3{add(F.lin.x, fw.x), add(F.lin.y, fw.y), add(F.lin.z, fw.z)};
        break;
    }
    case B200_EFF_GRAVITY_FRAME: { // falcon9/sim.py:350-361, frames.py:91-109
        const double mu = E.p[0];
        const Vec3 om = {E.p[1], E.p[2], E.p[3]};
        const Vec3 r = sx.x, v = sv.lin;
        const double rn = sqr(dot3(r));
        const double rn3 = mul(mul(rn, rn), rn);
        const Vec3 g = div3(Vec3{mul(-mu, r.x), mul(-mu, r.y), mul(-mu, r.z)}, rn3);
        const Vec3 c = cross(om, v);
        const Vec3 c2 = cross(om, cross(om, r));
        const Vec3 acc = {add(g.x, add(mul(-2.0, c.x), -c2.x)), add(g.y, add(mul(-2.0, c.y), -c2.y)),
                          add(g.z, add(mul(-2.0, c.z), -c2.z))};
        F.ang = Vec3{add(F.ang.x, 0.0), add(F.ang.y, 0.0), add(F.ang.z, 0.0)};
        F.lin = Vec3{add(F.lin.x, mul(acc.x, I.m)), add(F.lin.y, mul(acc.y, I.m)), add(F.lin.z, mul(acc.z, I.m))};
        break;
    }
    case B200_EFF_WRENCH_WORLD: { // cube-sat/main.py:516-527, drone/sim.py:99-103: force + SpatialForce(..)
        if (col()) {
            F.ang = Vec3{add(F.ang.x, ldp(col(), P.ld, 0, b)), add(F.ang.y, ldp(col(), P.ld, 1, b)), add(F.ang.z, ldp(col(), P.ld, 2, b))};
            F.lin = Vec3{add(F.lin.x, ldp(col(), P.ld, 3, b)), add(F.lin.y, ldp(col(), P.ld, 4, b)), add(F.lin.z, ldp(col(), P.ld, 5, b))};
        }
        break;
    }
    case B200_EFF_TORQUE_BODY_FOLD: { // cube-sat/main.py:492-505: Force := fold_k (f + SpatialForce(torque = q @ tau_k))
        if (col()) {
            Motion acc = {{0.0, 0.0, 0.0}, {0.0, 0.0, 0.0}};
            const uint32_t K = E.col_width / 3u;
            for (uint32_t k = 0; k < K; ++k) {
                const Vec3 t = qrot_with(sx.q, pi.qi, Vec3{ldp(col(), P.ld, 3 * k + 0, b), ldp(col(), P.ld, 3 * k + 1, b),
                                                           ldp(col(), P.ld, 3 * k + 2, b)});
                acc.ang = Vec3{add(acc.ang.x, t.x), add(acc.ang.y, t.y), add(acc.ang.z, t.z)};
                acc.lin = Vec3{add(acc.lin.x, 0.0), add(acc.lin.y, 0.0), add(acc.lin.z, 0.0)};
            }
            F = acc;
        }
        break;
    }
    case B200_EFF_GRAVITY_J2: { // python/elodin/j2.py:5-29
        const Vec3 g = j2_field_exact(E.p[0], E.p[1], E.p[2], sx.x, I.m);
        F.ang = Vec3{add(F.ang.x, 0.0), add(F.ang.y, 0.0), add(F.ang.z, 0.0)};
        F.lin = Vec3{add(F.lin.x, g.x), add(F.lin.y, g.y), add(F.lin.z, g.z)};
        break;
    }
    case B200_EFF_GRAVITY_EGM08: { // python/elodin/egm08.py; force + SpatialForce(linear=field): the field at this stage's
        if (P.aforce) {                // position was evaluated by egm08_force_kernel before this launch
            F.ang = Vec3{add(F.ang.x, 0.0), add(F.ang.y, 0.0), add(F.ang.z, 0.0)};
            F.lin = Vec3{add(F.lin.x, ldp(P.aforce, P.ld, slot * 3 + 0, b)), add(F.lin.y, ldp(P.aforce, P.ld, slot * 3 + 1, b)),
                         add(F.lin.z, ldp(P.aforce, P.ld, slot * 3 + 2, b))};
        }
        break;
    }
    case B200_EFF_GRAVITY_EDGES_NEWTON:
    case B200_EFF_GRAVITY_EDGES_SOFTENED: { // Force := edge_fold(init 0) for bodies that own an edge
        if (GREG) {
            if (greg.has) { F.ang = Vec3{0.0, 0.0, 0.0}; F.lin = grav_slot(greg, slot); }
        } else if (P.gforce && P.has_edge && P.has_edge[(b + P.ent0) % P.n_entities]) {
            F.ang = Vec3{0.0, 0.0, 0.0};
            F.lin = Vec3{ldp(P.gforce, P.ld, slot * 3 + 0, b), ldp(P.gforce, P.ld, slot * 3 + 1, b),
                         ldp(P.gforce, P.ld, slot * 3 + 2, b)};
        }
        break;
    }
    default: break;
    }
}

// clear_forces | effectors (array order) on the stage state; six_dof.rs:148-150,195
template <bool GREG, bool SCHED = false>
__device__ __forceinline__ Motion effectors_exact(const StepParams &P, uint64_t b, int slot, const Pose &sx,
                                                  const ex::PoseInv &pi, const Motion &sv, const Inertia &I,
                                                  const GravReg &greg, uint64_t tick = 0)
{
    Motion F = {{0.0, 0.0, 0.0}, {0.0, 0.0, 0.0}};
    for (uint32_t e = 0; e < P.n_eff; ++e) {
        const EffDev &E = P.eff[e];
        if (E.mask && !E.mask[(b + P.ent0) % P.n_entities]) continue; // entity does not own the effector's components (query join)
        apply_effector_exact<GREG, SCHED>(E.kind, E, P, b, slot, sx, pi, sv, I, greg, F, tick);
    }
    return F;
}

// The same pipe for an effector list known at compile time: SEQ packs the kinds of effectors 0..4 in list order, four
// bits each (0 ends the list; SEQ = 0 is the empty list).  Same operations in the same order as the interpreter — the
// order of accumulation is part of the arithmetic — without its loop, its switch, and the registers they pin.
static constexpr uint32_t SEQ_INTERPRET = 0xffffffffu;
template <uint32_t SEQ, bool GREG, bool SCHED = false>
__device__ __forceinline__ Motion effectors_exact_seq(const StepParams &P, uint64_t b, int slot, const Pose &sx,
                                                      const ex::PoseInv &pi, const Motion &sv, const Inertia &I,
                                                      const GravReg &greg, uint64_t tick = 0)
{
    Motion F = {{0.0, 0.0, 0.0}, {0.0, 0.0, 0.0}};
    if constexpr (((SEQ >> 0) & 15u) != 0) apply_effector_exact<GREG, SCHED>((SEQ >> 0) & 15u, P.eff[0], P, b, slot, sx, pi, sv, I, greg, F, tick);
    if constexpr (((SEQ >> 4) & 15u) != 0) apply_effector_exact<GREG, SCHED>((SEQ >> 4) & 15u, P.eff[1], P, b, slot, sx, pi, sv, I, greg, F, tick);
    if constexpr (((SEQ >> 8) & 15u) != 0) apply_effector_exact<GREG, SCHED>((SEQ >> 8) & 15u, P.eff[2], P, b, slot, sx, pi, sv, I, greg, F, tick);
    if constexpr (((SEQ >> 12) & 15u) != 0) apply_effector_exact<GREG, SCHED>((SEQ >> 12) & 15u, P.eff[3], P, b, slot, sx, pi, sv, I, greg, F, tick);
    if constexpr (((SEQ >> 16) & 15u) != 0) apply_effector_exact<GREG, SCHED>((SEQ >> 16) & 15u, P.eff[4], P, b, slot, sx, pi, sv, I, greg, F, tick);
    return F;
}

// one tick of one body in EXACT arithmetic (state in registers)
// UNR: unroll the three independent stage poses (more instruction-level parallelism across the dependent IEEE
// divisions, more registers) or keep them a loop
// SEQ: SEQ_INTERPRET = interpret P.eff[] at run time; anything else = the effector list as a compile-time sequence
// (0 = no effectors: clear_forces only)
// SCHED, tick: the launch carries input schedules, `tick` is the Tick column value of the tick integrated here
template <int INTEG, bool GREG, bool UNR = false, uint32_t SEQ = SEQ_INTERPRET, bool SCHED = false>
__device__ __forceinline__ void exact_tick(const StepParams &P, uint64_t b, Pose &x0, Motion &v0, Motion &a_out,
                                           Motion &f_out, const Inertia &I, const GravReg &greg, uint64_t tick = 0)
{
    using namespace ex;
    const InertiaRcp IR = inertia_rcp(I); // loop-invariant when a launch integrates several ticks
    if (INTEG == B200_INTEGRATOR_RK4) {
        // rk4.rs:85-123 (see the header comment of oracle/sixdof_oracle.c for the derivation)
        Motion sa = a_out; // du.a before stage 1 is the WorldAccel column
        Motion kv, ka;
        // three distinct stage poses (f = 0, .5, 1), functions of (x0, v0) only; stages 2 and 3 share
        // the f = .5 pose and its inverses — identical inputs, identical bits — so each is built once
#pragma unroll(UNR ? 3 : 1)
        for (int k = 0; k < 3; ++k) {
            const double dtf = mul(P.dt_stage, k == 0 ? 0.0 : (k == 1 ? 0.5 : 1.0));
            const Pose sx = tadd(x0, scale(dtf, v0));
            const PoseInv pi = pose_inverses(sx.q);
            const int n_stages = (k == 1) ? 2 : 1;
#pragma unroll 1
            for (int j = 0; j < n_stages; ++j) {
                const int s = (k == 0) ? 0 : (k == 1 ? 1 + j : 3);
                const Motion sv = madd(v0, scale(dtf, sa));
                if constexpr (SEQ == SEQ_INTERPRET) f_out = effectors_exact<GREG, SCHED>(P, b, k, sx, pi, sv, I, greg, tick);
                else f_out = effectors_exact_seq<SEQ, GREG, SCHED>(P, b, k, sx, pi, sv, I, greg, tick);
                sa = calc_accel_with(sx, pi, f_out, I, IR);
                if (s == 0) { kv = sv; ka = sa; }
                else if (s == 3) { kv = madd(kv, sv); ka = madd(ka, sa); }
                else { kv = madd(kv, scale(2.0, sv)); ka = madd(ka, scale(2.0, sa)); }
            }
        }
        const double c = mul(P.dt_final, 1.0 / 6.0);
        x0 = tadd(x0, scale(c, kv));
        v0 = madd(v0, scale(c, ka));
        a_out = sa;
    } else {
        // semi_implicit.rs:42-62
        const PoseInv pi = pose_inverses(x0.q);
        if constexpr (SEQ == SEQ_INTERPRET) f_out = effectors_exact<GREG, SCHED>(P, b, 0, x0, pi, v0, I, greg, tick);
        else f_out = effectors_exact_seq<SEQ, GREG, SCHED>(P, b, 0, x0, pi, v0, I, greg, tick);
        a_out = calc_accel_with(x0, pi, f_out, I, IR);
        v0 = madd(v0, scale(P.dt_final, a_out));
        x0 = tadd(x0, scale(P.dt_final, v0));
    }
}


// ================================================================== FAST ticks

// Compile-time effector signature of the specialised FAST kernels (SURVEY §2.4 K2: "template on an
// effector bitmask").  The host maps an effector list onto a signature when it can (body_kernels.cu:
// spec_signature); lists it cannot map (entity masks, repeated kinds, a wrench ahead of a drag) run
// through SIG_GENERIC, the run-time interpreter.  Constant gravity is part of every signature: its
// (summed) g sits in the constant bank and costs three multiplies.
enum : uint32_t {
    SIG_DRAG = 1u,            // DRAG_QUADRATIC with a wind column (width 3)
    SIG_DRAG_PB = 2u,         //   ... whose column also carries per-body [Cd*rho, area] (width 5)
    SIG_THRUST = 4u,          // THRUST_BODY
    SIG_WRENCH = 8u,          // WRENCH_BODY (either layout: the host hands over torque / force plane bases)
    SIG_FRAME = 16u,          // GRAVITY_FRAME
    SIG_GRAPH = 32u,          // GRAVITY_EDGES_*: 9 planes of edge_fold gravity
    SIG_J2 = 64u,             // GRAVITY_J2
    SIG_WHEELS = 128u,        // TORQUE_BODY_FOLD with three wheels (the cube-sat shape), first in the list
    SIG_WWORLD = 256u,        // WRENCH_WORLD: externally computed world-frame wrench column
    SIG_FREE = 512u,          // no effector and a summed constant gravity of exactly (0, 0, 0).  The tick is the sig-0
                              // arithmetic unchanged; only the kernel's velocity write-back differs (no effector code
                              // tests this bit)
    SIG_GENERIC = 0x80000000u // interpret StepParams::eff[] at run time
};

// The inertia diagonal enters the tick only through invI, which only body-frame and world-frame torques need
__host__ __device__ constexpr bool sig_needs_invI(uint32_t sig)
{
    return sig == SIG_GENERIC || (sig & (SIG_WRENCH | SIG_WHEELS | SIG_WWORLD)) != 0;
}

// per-body effector inputs of a specialised kernel: loaded next to the state, before any arithmetic
struct EffIn {
    double thrust;
    Vec3 wr_t, wr_f; // body-frame torque / force of the wrench column
    Vec3 wind;
    double cd_rho, area;
    Vec3 wheels;     // sum of the body's wheel torques (body frame)
    Vec3 ww_t, ww_f; // world-frame torque / force of the WRENCH_WORLD column
};

// Everything the effector list contributes, folded once per launch:
//   F_lin(stage) = fw + R(q) fb + drag(v) + m*frame(x, v) + gforce[slot]
//   a_ang(stage) = R(q) u,   u = (sum of body-frame torques) / diag(I)   (R^-1 then R cancel)
struct Folded {
    Vec3 fw;      // world-frame constant force (GRAVITY_CONST: g*m)
    Vec3 fb;      // body-frame force (THRUST_BODY axis*thrust, WRENCH_BODY force part)
    Vec3 u;       // body-frame angular acceleration
    Vec3 wind;    // DRAG_QUADRATIC
    double kd;    // 0.5*Cd*rho*A
    double mu;    // GRAVITY_FRAME
    Vec3 om;
    Vec3 tw;      // world-frame torque (WRENCH_WORLD): needs R^-1 per stage attitude
    double j2_mu, j2_k; // GRAVITY_J2: mu, J2 * r_ref^2
    bool drag, frame, graph, wtorque, j2;
    bool aforce;        // GRAVITY_EGM08: add the stage-force planes egm08_force_kernel filled
};

// SCHED: the launch carries input schedules; effector columns are read at the row of `tick`
template <bool GREG, bool SCHED = false>
__device__ __forceinline__ Folded fold_effectors(const StepParams &P, uint64_t b, const Inertia &I, const Vec3 &invI,
                                                 const GravReg &greg, uint64_t tick = 0)
{
    Folded f;
    f.fw = f.fb = f.u = f.wind = f.om = Vec3{0.0, 0.0, 0.0};
    f.kd = f.mu = f.j2_mu = f.j2_k = 0.0;
    f.tw = Vec3{0.0, 0.0, 0.0};
    f.drag = f.frame = f.graph = f.wtorque = f.j2 = f.aforce = false;
    Vec3 tb = {0.0, 0.0, 0.0};
    for (uint32_t e = 0; e < P.n_eff; ++e) {
        const EffDev &E = P.eff[e];
        if (E.mask && !E.mask[(b + P.ent0) % P.n_entities]) continue; // query join: not a member
        auto col = [&]() { return SCHED ? schedule_ptr(E.col, E.sched, tick) : E.col; }; // read at each use, like E.col
        switch (E.kind) {
        case B200_EFF_GRAVITY_CONST:
            f.fw.x = fma(E.p[0], I.m, f.fw.x); f.fw.y = fma(E.p[1], I.m, f.fw.y); f.fw.z = fma(E.p[2], I.m, f.fw.z);
            break;
        case B200_EFF_DRAG_QUADRATIC:
            f.drag = true;
            f.kd = E.col_width == 5 ? 0.5 * ldp(col(), P.ld, 3, b) * ldp(col(), P.ld, 4, b) : 0.5 * E.p[0] * E.p[1];
            if (col()) f.wind = Vec3{ldp(col(), P.ld, 0, b), ldp(col(), P.ld, 1, b), ldp(col(), P.ld, 2, b)};
            tb = Vec3{0.0, 0.0, 0.0}; // the reference's apply_drag returns SpatialForce(linear=...): torque reset
            break;
        case B200_EFF_THRUST_BODY: {
            const double t = col() ? ldp(col(), P.ld, 0, b) : 0.0;
            f.fb.x = fma(E.p[0], t, f.fb.x); f.fb.y = fma(E.p[1], t, f.fb.y); f.fb.z = fma(E.p[2], t, f.fb.z);
            break;
        }
        case B200_EFF_WRENCH_BODY:
            if (col()) {
                const int to = (E.flags & B200_EFF_FLAG_WRENCH_LINEAR_FIRST) ? 3 : 0;
                const int fo = 3 - to;
                tb.x += ldp(col(), P.ld, to + 0, b); tb.y += ldp(col(), P.ld, to + 1, b); tb.z += ldp(col(), P.ld, to + 2, b);
                f.fb.x += ldp(col(), P.ld, fo + 0, b); f.fb.y += ldp(col(), P.ld, fo + 1, b); f.fb.z += ldp(col(), P.ld, fo + 2, b);
            }
            break;
        case B200_EFF_GRAVITY_FRAME:
            f.frame = true;
            f.mu = E.p[0];
            f.om = Vec3{E.p[1], E.p[2], E.p[3]};
            break;
        case B200_EFF_WRENCH_WORLD:
            if (col()) {
                f.tw.x += ldp(col(), P.ld, 0, b); f.tw.y += ldp(col(), P.ld, 1, b); f.tw.z += ldp(col(), P.ld, 2, b);
                f.fw.x += ldp(col(), P.ld, 3, b); f.fw.y += ldp(col(), P.ld, 4, b); f.fw.z += ldp(col(), P.ld, 5, b);
                f.wtorque = true;
            }
            break;
        case B200_EFF_TORQUE_BODY_FOLD: // Force := fold: everything accumulated before it is overwritten
            if (col()) {
                tb = Vec3{0.0, 0.0, 0.0};
                f.fw = f.fb = f.tw = Vec3{0.0, 0.0, 0.0};
                f.drag = f.frame = f.wtorque = f.j2 = f.aforce = false;
                const uint32_t K = E.col_width / 3u;
                for (uint32_t k = 0; k < K; ++k) {
                    tb.x += ldp(col(), P.ld, 3 * k + 0, b); tb.y += ldp(col(), P.ld, 3 * k + 1, b); tb.z += ldp(col(), P.ld, 3 * k + 2, b);
                }
            }
            break;
        case B200_EFF_GRAVITY_J2:
            f.j2 = true;
            f.j2_mu = E.p[0];
            f.j2_k = E.p[1] * E.p[2] * E.p[2];
            break;
        case B200_EFF_GRAVITY_EGM08:
            f.aforce = P.aforce != nullptr;
            break;
        case B200_EFF_GRAVITY_EDGES_NEWTON:
        case B200_EFF_GRAVITY_EDGES_SOFTENED: // host guarantees this is effector 0 in FAST mode
            f.graph = GREG ? greg.has : (P.gforce && P.has_edge && P.has_edge[(b + P.ent0) % P.n_entities]);
            break;
        default: break;
        }
    }
    f.u = Vec3{tb.x * invI.x, tb.y * invI.y, tb.z * invI.z};
    return f;
}

// the per-body inputs of signature SIG at the schedule rows of `tick` (fused launches with input schedules: every tick
// after the first reloads them; the first tick's inputs arrive with the state loads)
template <uint32_t SIG>
__device__ __forceinline__ EffIn load_spec_inputs(const StepParams &P, uint64_t b, uint64_t tick)
{
    EffIn in;
    in.thrust = 0.0; in.cd_rho = in.area = 0.0;
    in.wr_t = in.wr_f = in.wind = in.wheels = in.ww_t = in.ww_f = Vec3{0.0, 0.0, 0.0};
    if (SIG & SIG_THRUST) in.thrust = ldp(schedule_ptr(P.spec.thrust, P.spec.s_thrust, tick), P.ld, 0, b);
    if (SIG & SIG_WRENCH) {
        const double *t = schedule_ptr(P.spec.wr_t, P.spec.s_wrench, tick), *f = schedule_ptr(P.spec.wr_f, P.spec.s_wrench, tick);
        in.wr_t = Vec3{ldp(t, P.ld, 0, b), ldp(t, P.ld, 1, b), ldp(t, P.ld, 2, b)};
        in.wr_f = Vec3{ldp(f, P.ld, 0, b), ldp(f, P.ld, 1, b), ldp(f, P.ld, 2, b)};
    }
    if (SIG & SIG_WHEELS) { // summed in the order the kernel's initial load sums them
        const double *w = schedule_ptr(P.spec.wheels, P.spec.s_wheels, tick);
        in.wheels = Vec3{ldp(w, P.ld, 0, b) + ldp(w, P.ld, 3, b) + ldp(w, P.ld, 6, b), ldp(w, P.ld, 1, b) + ldp(w, P.ld, 4, b) + ldp(w, P.ld, 7, b),
                         ldp(w, P.ld, 2, b) + ldp(w, P.ld, 5, b) + ldp(w, P.ld, 8, b)};
    }
    if (SIG & SIG_WWORLD) {
        const double *w = schedule_ptr(P.spec.wworld, P.spec.s_wworld, tick);
        in.ww_t = Vec3{ldp(w, P.ld, 0, b), ldp(w, P.ld, 1, b), ldp(w, P.ld, 2, b)};
        in.ww_f = Vec3{ldp(w, P.ld, 3, b), ldp(w, P.ld, 4, b), ldp(w, P.ld, 5, b)};
    }
    if (SIG & SIG_DRAG) {
        const double *d = schedule_ptr(P.spec.drag, P.spec.s_drag, tick);
        in.wind = Vec3{ldp(d, P.ld, 0, b), ldp(d, P.ld, 1, b), ldp(d, P.ld, 2, b)};
        if (SIG & SIG_DRAG_PB) { in.cd_rho = ldp(d, P.ld, 3, b); in.area = ldp(d, P.ld, 4, b); }
    }
    return in;
}

// the same fold for a compile-time signature: constants from StepParams::spec (constant bank), per-body inputs
// from registers; members the signature does not use are literal zeros the optimiser removes
template <uint32_t SIG, bool GREG>
__device__ __forceinline__ Folded fold_spec(const StepParams &P, uint64_t b, const EffIn &in, const Inertia &I, const Vec3 &invI,
                                            const GravReg &greg)
{
    Folded f;
    f.fw = Vec3{P.spec.g[0] * I.m, P.spec.g[1] * I.m, P.spec.g[2] * I.m};
    f.fb = f.u = f.wind = f.om = Vec3{0.0, 0.0, 0.0};
    f.kd = f.mu = f.j2_mu = f.j2_k = 0.0;
    f.tw = Vec3{0.0, 0.0, 0.0};
    f.wtorque = f.j2 = f.aforce = false;
    f.drag = (SIG & SIG_DRAG) != 0;
    f.frame = (SIG & SIG_FRAME) != 0;
    f.graph = (SIG & SIG_GRAPH) ? (GREG ? greg.has : P.has_edge[(b + P.ent0) % P.n_entities] != 0) : false;
    if (SIG & SIG_THRUST) f.fb = Vec3{P.spec.axis[0] * in.thrust, P.spec.axis[1] * in.thrust, P.spec.axis[2] * in.thrust};
    Vec3 tb = {0.0, 0.0, 0.0};
    if (SIG & SIG_WHEELS) tb = in.wheels;
    if (SIG & SIG_WRENCH) {
        f.fb = Vec3{f.fb.x + in.wr_f.x, f.fb.y + in.wr_f.y, f.fb.z + in.wr_f.z};
        tb = Vec3{tb.x + in.wr_t.x, tb.y + in.wr_t.y, tb.z + in.wr_t.z};
    }
    if (SIG & (SIG_WRENCH | SIG_WHEELS)) f.u = Vec3{tb.x * invI.x, tb.y * invI.y, tb.z * invI.z};
    if (SIG & SIG_J2) {
        f.j2 = true;
        f.j2_mu = P.spec.j2_mu;
        f.j2_k = P.spec.j2_k;
    }
    if (SIG & SIG_WWORLD) {
        f.fw = Vec3{f.fw.x + in.ww_f.x, f.fw.y + in.ww_f.y, f.fw.z + in.ww_f.z};
        f.tw = in.ww_t;
        f.wtorque = true;
    }
    if (SIG & SIG_DRAG) {
        f.wind = in.wind;
        f.kd = (SIG & SIG_DRAG_PB) ? 0.5 * in.cd_rho * in.area : P.spec.kd;
    }
    if (SIG & SIG_FRAME) {
        f.mu = P.spec.mu;
        f.om = Vec3{P.spec.om[0], P.spec.om[1], P.spec.om[2]};
    }
    return f;
}

// linear acceleration of one stage: everything that depends on (q, x, v)
template <bool GREG>
__device__ __forceinline__ Vec3 lin_accel_fast(const StepParams &P, const Folded &f, uint64_t b, int slot,
                                               const Vec3 &fbw, const Vec3 &x, const Vec3 &v, double m, double inv_m,
                                               const GravReg &greg)
{
    Vec3 F = {f.fw.x + fbw.x, f.fw.y + fbw.y, f.fw.z + fbw.z};
    if (f.drag) {
        const Vec3 fl = {f.wind.x - v.x, f.wind.y - v.y, f.wind.z - v.z};
        const double s2 = fl.x * fl.x + fl.y * fl.y + fl.z * fl.z;
        // drag*dir = (kd*speed^2) * fl/speed = kd*speed*fl, speed = s2 * rsqrt(s2); speed == 0 gives 0 * inf = NaN
        // like the reference's 0/0
        const double k = f.kd * (s2 * fa::rsqrt_nr(s2));
        F.x = fma(k, fl.x, F.x); F.y = fma(k, fl.y, F.y); F.z = fma(k, fl.z, F.z);
    }
    if (f.frame) {
        const double r2 = x.x * x.x + x.y * x.y + x.z * x.z;
        const double ir = fa::rsqrt_nr(r2);
        const double g = -f.mu * ir * ir * ir;
        const Vec3 c = fa::cross(f.om, v);
        const Vec3 c2 = fa::cross(f.om, fa::cross(f.om, x));
        F.x = fma(fma(g, x.x, -2.0 * c.x - c2.x), m, F.x);
        F.y = fma(fma(g, x.y, -2.0 * c.y - c2.y), m, F.y);
        F.z = fma(fma(g, x.z, -2.0 * c.z - c2.z), m, F.z);
    }
    if (f.j2) {
        // -mu m [ r/n^3 + J2 r_ref^2 ( 3 z/n^5 e_z + (3/(2 n^4) - 15 z^2/(2 n^6)) r/n ) ]   (j2.py:12-27)
        const double r2 = x.x * x.x + x.y * x.y + x.z * x.z;
        const double ir = fa::rsqrt_nr(r2), ir2 = ir * ir, ir3 = ir2 * ir, ir5 = ir3 * ir2;
        const double kr = f.j2_k * ir5 * (1.5 - 7.5 * x.z * x.z * ir2); // coefficient of r (e_r = r/n folded in)
        const double kz = 3.0 * f.j2_k * x.z * ir5;
        const double c = -f.j2_mu * m;
        F.x = fma(c, (ir3 + kr) * x.x, F.x);
        F.y = fma(c, (ir3 + kr) * x.y, F.y);
        F.z = fma(c, fma(ir3 + kr, x.z, kz), F.z);
    }
    if (f.aforce) { // the harmonic series at this stage's position, evaluated by egm08_force_kernel with the oracle's arithmetic
        F.x += ldp(P.aforce, P.ld, slot * 3 + 0, b);
        F.y += ldp(P.aforce, P.ld, slot * 3 + 1, b);
        F.z += ldp(P.aforce, P.ld, slot * 3 + 2, b);
    }
    if (f.graph) {
        if (GREG) {
            const Vec3 g = grav_slot(greg, slot);
            F.x += g.x; F.y += g.y; F.z += g.z;
        } else {
            F.x += ldp(P.gforce, P.ld, slot * 3 + 0, b);
            F.y += ldp(P.gforce, P.ld, slot * 3 + 1, b);
            F.z += ldp(P.gforce, P.ld, slot * 3 + 2, b);
        }
    }
    return Vec3{F.x * inv_m, F.y * inv_m, F.z * inv_m};
}

// world-frame force this stage's state produced (only materialised when Force is written back)
__device__ __forceinline__ Motion force_out_fast(const Vec3 &a_lin, const Vec3 &a_ang_body_u, const Quat &q,
                                                 const Inertia &I, const Vec3 &tw)
{
    // torque_world = R (I .* u) + the world-frame torque column
    const Vec3 tb = {a_ang_body_u.x * I.diag.x, a_ang_body_u.y * I.diag.y, a_ang_body_u.z * I.diag.z};
    Motion F;
    F.ang = fa::rot(q, tb);
    F.ang = Vec3{F.ang.x + tw.x, F.ang.y + tw.y, F.ang.z + tw.z};
    F.lin = Vec3{a_lin.x * I.m, a_lin.y * I.m, a_lin.z * I.m};
    return F;
}

// n_ticks ticks of one body, state in registers (shared by the direct and the TMA-pipelined kernel)
// (n_ticks, tick0, want_f) are P.n_ticks, P.tick0, P.write_fa for the kernels that integrate a launch's ticks
// in one call; small_world_kernel calls it once per tick with that tick's gravity in `greg`
// SCHED: the launch carries input schedules (P.sched): tick t of the launch (Tick value P.tick_abs + t) folds the
// effector inputs of its own schedule rows; `in` holds the first tick's
template <int INTEG, bool TRAJ, bool GREG = false, uint32_t SIG = SIG_GENERIC, bool SCHED = false>
__device__ __forceinline__ void fast_ticks(const StepParams &P, uint64_t b, Pose &x0, Motion &v0, const Inertia &I,
                                           Motion &a_last, Motion &f_last, uint32_t n_ticks, uint64_t tick0, bool want_f,
                                           const GravReg &greg, const EffIn &in = EffIn{}, bool store_traj = true)
{
    constexpr bool GEN = SIG == SIG_GENERIC;
    constexpr bool NEED_INVI = sig_needs_invI(SIG);
    const Vec3 invI = NEED_INVI ? Vec3{fa::rcp_nr(I.diag.x), fa::rcp_nr(I.diag.y), fa::rcp_nr(I.diag.z)} : Vec3{0.0, 0.0, 0.0};
    const double inv_m = fa::rcp_nr(I.m);
    Folded f;
    if constexpr (GEN) f = fold_effectors<GREG, SCHED>(P, b, I, invI, greg, P.tick_abs);
    else f = fold_spec<SIG, GREG>(P, b, in, I, invI, greg);

    a_last = Motion{{0.0, 0.0, 0.0}, {0.0, 0.0, 0.0}};
    Quat q_last = x0.q;
    const double dt = P.dt_stage;
    // generic: data-dependent (most bodies of a heterogeneous world carry no body-frame wrench; NaNs compare
    // unequal to zero and take the full path); specialised: a property of the signature
    // (a scheduled interpreter launch re-derives them with every tick's fold)
    bool has_u = GEN ? ((f.u.x != 0.0) | (f.u.y != 0.0) | (f.u.z != 0.0)) : (SIG & (SIG_WRENCH | SIG_WHEELS)) != 0;
    bool has_fb = GEN ? ((f.fb.x != 0.0) | (f.fb.y != 0.0) | (f.fb.z != 0.0)) : (SIG & (SIG_THRUST | SIG_WRENCH)) != 0;
    bool has_tw = GEN ? f.wtorque : (SIG & SIG_WWORLD) != 0; // world-frame torque: a_ang = R (invI .* (R^-1 tau_w)) per stage attitude
    auto ang_world = [&](const Quat &q) { // angular acceleration the world-frame torque produces at attitude q
        const Vec3 tbody = fa::rot(Quat{-q.i, -q.j, -q.k, q.w}, f.tw);
        return fa::rot(q, Vec3{tbody.x * invI.x, tbody.y * invI.y, tbody.z * invI.z});
    };

    // telemetry samples: one 64-bit division per call instead of one per tick (a sample is due when the tick count
    // reaches a multiple of traj_every; its slot is that multiple's index - 1)
    uint32_t traj_phase = 0;
    uint64_t traj_slot = 0;
    if (TRAJ && P.traj_every) { traj_phase = (uint32_t)(tick0 % P.traj_every); traj_slot = tick0 / P.traj_every; }

    for (uint32_t t = 0; t < n_ticks; ++t) {
        if constexpr (SCHED) {
            if (t > 0) {
                if constexpr (GEN) {
                    f = fold_effectors<GREG, true>(P, b, I, invI, greg, P.tick_abs + t);
                    has_u = (f.u.x != 0.0) | (f.u.y != 0.0) | (f.u.z != 0.0);
                    has_fb = (f.fb.x != 0.0) | (f.fb.y != 0.0) | (f.fb.z != 0.0);
                    has_tw = f.wtorque;
                } else {
                    f = fold_spec<SIG, GREG>(P, b, load_spec_inputs<SIG>(P, b, P.tick_abs + t), I, invI, greg);
                }
            }
        }
        if (INTEG == B200_INTEGRATOR_RK4) {
            const Vec3 w0 = v0.ang, u0 = v0.lin;
            // the three distinct stage poses depend on (x0, v0) only (rk4.rs:85-111)
            // (the stage attitudes only matter to bodies that carry a body-frame force or torque)
            const double h2 = 0.25 * dt, h4 = 0.5 * dt;
            Quat q1 = x0.q, q2 = x0.q, q4 = x0.q;
            if (has_u | has_fb | has_tw) {
                q1 = fa::normalize(x0.q); // x0 (+) 0*v0 still renormalises (spatial.rs:540-545)
                q2 = fa::advance(x0.q, Vec3{h2 * w0.x, h2 * w0.y, h2 * w0.z});
                q4 = fa::advance(x0.q, Vec3{h4 * w0.x, h4 * w0.y, h4 * w0.z});
            }
            const Vec3 x2 = {fma(h4, u0.x, x0.x.x), fma(h4, u0.y, x0.x.y), fma(h4, u0.z, x0.x.z)};
            const Vec3 x4 = {fma(dt, u0.x, x0.x.x), fma(dt, u0.y, x0.x.y), fma(dt, u0.z, x0.x.z)};
            // angular acceleration R(q) u and rotated body force, once per distinct attitude
            const Vec3 zero3 = {0.0, 0.0, 0.0};
            Vec3 aa1 = zero3, aa2 = zero3, aa4 = zero3, fb1 = zero3, fb2 = zero3, fb4 = zero3;
            if (has_u) { aa1 = fa::rot(q1, f.u); aa2 = fa::rot(q2, f.u); aa4 = fa::rot(q4, f.u); }
            if (has_fb) { fb1 = fa::rot(q1, f.fb); fb2 = fa::rot(q2, f.fb); fb4 = fa::rot(q4, f.fb); }
            if (has_tw) {
                const Vec3 w1 = ang_world(q1), w2 = ang_world(q2), w4 = ang_world(q4);
                aa1 = Vec3{aa1.x + w1.x, aa1.y + w1.y, aa1.z + w1.z};
                aa2 = Vec3{aa2.x + w2.x, aa2.y + w2.y, aa2.z + w2.z};
                aa4 = Vec3{aa4.x + w4.x, aa4.y + w4.y, aa4.z + w4.z};
            }
            // stage 1: v = v0
            const Vec3 al1 = lin_accel_fast<GREG>(P, f, b, 0, fb1, x0.x, u0, I.m, inv_m, greg);
            // stage 2: v = v0 + dt/2 a1
            const Vec3 u2 = {fma(h4, al1.x, u0.x), fma(h4, al1.y, u0.y), fma(h4, al1.z, u0.z)};
            const Vec3 al2 = lin_accel_fast<GREG>(P, f, b, 1, fb2, x2, u2, I.m, inv_m, greg);
            // stage 3: same pose as stage 2, v = v0 + dt/2 a2
            const Vec3 u3 = {fma(h4, al2.x, u0.x), fma(h4, al2.y, u0.y), fma(h4, al2.z, u0.z)};
            const Vec3 al3 = lin_accel_fast<GREG>(P, f, b, 1, fb2, x2, u3, I.m, inv_m, greg);
            // stage 4: v = v0 + dt a3
            const Vec3 u4 = {fma(dt, al3.x, u0.x), fma(dt, al3.y, u0.y), fma(dt, al3.z, u0.z)};
            const Vec3 al4 = lin_accel_fast<GREG>(P, f, b, 2, fb4, x4, u4, I.m, inv_m, greg);
            // k.v sum = 6 v0 + dt (a1 + a2 + a3);  k.a sum = a1 + 2 a2 + 2 a3 + a4   (a3.ang == a2.ang)
            const double c = P.dt_final * (1.0 / 6.0);
            const Vec3 kw = {fma(dt, aa1.x + 2.0 * aa2.x, 6.0 * w0.x), fma(dt, aa1.y + 2.0 * aa2.y, 6.0 * w0.y),
                             fma(dt, aa1.z + 2.0 * aa2.z, 6.0 * w0.z)};
            const Vec3 ku = {fma(dt, al1.x + al2.x + al3.x, 6.0 * u0.x), fma(dt, al1.y + al2.y + al3.y, 6.0 * u0.y),
                             fma(dt, al1.z + al2.z + al3.z, 6.0 * u0.z)};
            const double hc = 0.5 * c;
            x0.q = fa::advance(x0.q, Vec3{hc * kw.x, hc * kw.y, hc * kw.z});
            x0.x = Vec3{fma(c, ku.x, x0.x.x), fma(c, ku.y, x0.x.y), fma(c, ku.z, x0.x.z)};
            v0.ang = Vec3{fma(c, aa1.x + 4.0 * aa2.x + aa4.x, w0.x), fma(c, aa1.y + 4.0 * aa2.y + aa4.y, w0.y),
                          fma(c, aa1.z + 4.0 * aa2.z + aa4.z, w0.z)};
            v0.lin = Vec3{fma(c, al1.x + 2.0 * (al2.x + al3.x) + al4.x, u0.x),
                          fma(c, al1.y + 2.0 * (al2.y + al3.y) + al4.y, u0.y),
                          fma(c, al1.z + 2.0 * (al2.z + al3.z) + al4.z, u0.z)};
            a_last.ang = aa4; a_last.lin = al4; q_last = q4;
        } else {
            // semi_implicit.rs:42-62; calc_accel rotates by q/|q| whatever |q| is
            const double n2 = x0.q.i * x0.q.i + x0.q.j * x0.q.j + x0.q.k * x0.q.k + x0.q.w * x0.q.w;
            const double rn = fa::rsqrt_nr(n2);
            const Quat qn = {x0.q.i * rn, x0.q.j * rn, x0.q.k * rn, x0.q.w * rn};
            Vec3 aa = has_u ? fa::rot(qn, f.u) : Vec3{0.0, 0.0, 0.0};
            if (has_tw) { const Vec3 w = ang_world(qn); aa = Vec3{aa.x + w.x, aa.y + w.y, aa.z + w.z}; }
            const Vec3 fbw = has_fb ? fa::rot(qn, f.fb) : Vec3{0.0, 0.0, 0.0};
            const Vec3 al = lin_accel_fast<GREG>(P, f, b, 0, fbw, x0.x, v0.lin, I.m, inv_m, greg);
            const double d = P.dt_final;
            v0.ang = Vec3{fma(d, aa.x, v0.ang.x), fma(d, aa.y, v0.ang.y), fma(d, aa.z, v0.ang.z)};
            v0.lin = Vec3{fma(d, al.x, v0.lin.x), fma(d, al.y, v0.lin.y), fma(d, al.z, v0.lin.z)};
            const double hd = 0.5 * d;
            x0.q = fa::advance(x0.q, Vec3{hd * v0.ang.x, hd * v0.ang.y, hd * v0.ang.z});
            x0.x = Vec3{fma(d, v0.lin.x, x0.x.x), fma(d, v0.lin.y, x0.x.y), fma(d, v0.lin.z, x0.x.z)};
            a_last.ang = aa; a_last.lin = al; q_last = qn;
        }
        if (TRAJ && P.traj_every && store_traj) { // compiled out of the launches that record nothing (the roofline case)
            if (++traj_phase == P.traj_every) {
                traj_phase = 0;
                if (traj_slot < P.traj_capacity) {
                    traj_store_state(P, b, traj_slot, x0, v0);
                    if (P.traj_planes == 25) traj_store_af(P, b, traj_slot, a_last, force_out_fast(a_last.lin, f.u, q_last, I, f.tw));
                }
                ++traj_slot;
            }
        }
    }
    if (want_f) f_last = force_out_fast(a_last.lin, f.u, q_last, I, f.tw);
}

} // namespace b200
