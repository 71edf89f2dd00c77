// Host<->kernel parameter blocks of libb200_sixdof (internal; the public surface
// is include/b200_sixdof.h).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "../../include/b200_sixdof.h"

namespace b200 {

// Row of an input schedule (b200_sixdof_set_schedule) that the tick whose Tick column value is `tick` reads: the
// first row before the table starts, the last one after it ends.  The one place the rule lives (host and device).
__host__ __device__ __forceinline__ uint64_t schedule_row(uint64_t tick, uint64_t first_tick, uint64_t n_rows)
{
    const uint64_t r = tick > first_tick ? tick - first_tick : 0;
    return r < n_rows ? r : n_rows - 1;
}

// A scheduled column as a fused launch sees it: row r of the table starts `stride` doubles after row r-1 (width*ld,
// each row laid out like the column itself); stride 0 = not scheduled, the base is the column (or one fixed row).
struct SchedDev {
    uint64_t stride;
    uint64_t n_rows;
    uint64_t first_tick;
};
__host__ __device__ __forceinline__ const double *schedule_ptr(const double *base, const SchedDev &s, uint64_t tick)
{
    return s.stride ? base + schedule_row(tick, s.first_tick, s.n_rows) * s.stride : base;
}

// One built-in effector as the kernels see it.  `col` points at the SoA planes
// of its per-body input column (plane p at col + p*ld), nullptr if none.
struct EffDev {
    uint32_t kind;
    uint32_t flags;
    double p[8];
    const double *col;
    uint32_t col_width;
    uint32_t pad;
    const uint8_t *mask; // [n_entities] or nullptr (query-join membership)
    const double *table; // GRAVITY_EGM08: the term stream sixdof_abi.cu:egm08_tables builds (device)
    SchedDev sched;      // fused launches of a scheduled column: `col` is the table, tick t reads its row
};

// Launch parameters of the per-body integrator kernels.  All columns are SoA:
// plane k of a column lives at base + k*ld, body b at [.. + b].
struct StepParams {
    double *pos;        // 7 planes: q.i q.j q.k q.w x y z
    double *vel;        // 6 planes: omega(3) v(3)
    double *acc;        // 6 planes (WorldAccel; stage-4 value on output)
    double *frc;        // 6 planes (Force; stage-4 value on output)
    const double *ine;  // 7 planes: diag(3) momentum(3) mass
    const double *gforce; // 9 planes: edge_fold gravity at the 3 distinct stage positions (or nullptr)
    const uint8_t *has_edge; // [n_entities]: body owns >= 1 out-edge (or nullptr)
    const double *aforce;    // 9 planes: additive stage forces (GRAVITY_EGM08) at the 3 distinct stage positions (or nullptr)
    uint64_t ld;        // plane stride in doubles
    uint64_t n_bodies;  // n_worlds * n_entities
    uint32_t n_entities;
    uint32_t n_eff;
    double dt_stage;    // SimulationTimeStep (rk4.rs:90)
    double dt_final;    // six_dof(time_step=) or dt_stage (rk4.rs:83,119)
    uint32_t n_ticks;   // ticks integrated by this launch (state stays in registers)
    uint32_t write_fa;  // materialise Force / WorldAccel at the end of the launch
    // trajectory ring: sample s, plane p at traj + (s*traj_planes + p)*ld
    double *traj;
    uint64_t traj_capacity;
    uint32_t traj_every;  // 0 = off
    uint32_t traj_planes; // 13 (pos, vel) or 25 (+ accel, force)
    uint64_t tick0;     // global tick count before this launch
    uint32_t ent0;      // entity row of body 0 of this launch (row-sharded single worlds start inside a world)
    uint32_t reverse;   // walk the tiles from the last one down (alternating launches: L2 reuse of the previous launch's tail)
    // compile-time-specialised FAST kernels (sixdof_tick.cuh SIG_*): what body_kernels.cu:spec_signature
    // distilled from eff[] — uniform constants and the plane bases of the per-body input columns
    struct Spec {
        double g[3];        // sum of the GRAVITY_CONST vectors
        double axis[3];     // THRUST_BODY body axis
        double kd;          // 0.5 * Cd*rho * area of a DRAG_QUADRATIC without per-body parameters
        double mu, om[3];   // GRAVITY_FRAME
        double j2_mu, j2_k; // GRAVITY_J2: mu, J2 * r_ref^2
        const double *wheels;        // 9 planes: three body-frame wheel torques
        const double *wworld;        // 6 planes: world-frame wrench [tau, f]
        const double *thrust;        // 1 plane
        const double *wr_t, *wr_f;   // 3 planes each: body-frame torque / force of the wrench column
        const double *drag;          // wind(3) [+ Cd*rho, area]
        SchedDev s_wheels, s_wworld, s_thrust, s_wrench, s_drag; // the schedules of those columns (stride 0: none)
    } spec;
    EffDev eff[B200_MAX_EFFECTORS];
    uint64_t tick_abs;  // Tick column value of this launch's first tick (input schedules; tick0 restarts at a trajectory reset)
    uint32_t sched;     // some eff[].sched is live: the launch integrates > 1 tick and each tick reads its own row
    uint32_t pad_sched;
};

// Launch parameters of the edge_fold gravity kernels.
struct GraphParams {
    const double *pos, *vel, *ine;
    double *gforce;          // 9 planes out
    uint64_t ld;
    uint32_t n_entities;
    uint32_t n_worlds;
    double dt_stage;
    uint32_t kind;           // B200_EFF_GRAVITY_EDGES_*
    uint32_t integrator;     // B200_INTEGRATOR_*: RK4 evaluates 3 stage positions, semi-implicit 1
    double p0, p1;           // G | K^2, softening
    const uint32_t *row_ptr; // CSR over sources (n_entities+1), spawn order kept inside a row
    const uint32_t *col_idx;
    uint32_t max_deg;        // largest out-degree (uniform trip count of small_world_kernel's shuffle loop)
    uint32_t src0;           // dense kernels: fold only the source rows [src0, src0 + src_n) of every world (row-sharded
    uint32_t src_n;          // single worlds); src_n = 0 means every source
    uint32_t pad;
};

// Column table of the one-launch layout kernel used by small batches
struct MultiColumns {
    struct Col {
        uint64_t aos_offset; // doubles from `packed`
        double *soa;         // plane 0 of the device column
        uint32_t width;
        uint32_t pad;
    };
    double *packed;          // packed AoS staging (device)
    uint32_t n;
    uint32_t pad;
    Col col[16];
};

// kernel launchers (sixdof_kernels.cu); every one returns the launch status
cudaError_t launch_body_step(const StepParams &P, int integrator, int math_mode, cudaStream_t s);
cudaError_t launch_graph_force(const GraphParams &G, int math_mode, bool dense, cudaStream_t s);
// one-launch n-body tick (gravity + integration) for small grids; new pose / velocity go to *_out
bool nbody_fused_applicable(const GraphParams &G, int math_mode, bool dense);
cudaError_t launch_nbody_tick_fused(const GraphParams &G, const StepParams &P, double *pos_out, double *vel_out, cudaStream_t s);
// worlds of <= 32 bodies: gravity + integration of n_ticks ticks in one launch, one warp per floor(32/N) worlds
bool small_world_applicable(const GraphParams &G, int math_mode);
cudaError_t launch_small_world(const GraphParams &G, const StepParams &P, int math_mode, cudaStream_t s);
// GRAVITY_EGM08: the field at the three stage positions of every body -> 9 planes (one launch per tick)
struct EgmParams {
    const double *pos, *vel, *ine;
    double *aforce;
    const double *table;     // term stream of sixdof_abi.cu:egm08_tables (device)
    const uint8_t *mask;     // entity mask of the effector or nullptr
    uint64_t ld, n_bodies;
    uint32_t n_entities, ent0;
    uint32_t L, integrator;
    double mu, r_ref, dt_stage;
};
cudaError_t launch_egm08_force(const EgmParams &E, int math_mode, cudaStream_t s);
cudaError_t launch_aos_to_soa(const double *aos, double *soa, uint64_t n_bodies, uint32_t width, uint64_t ld,
                              cudaStream_t s);
cudaError_t launch_soa_to_aos(const double *soa, double *aos, uint64_t n_bodies, uint32_t width, uint64_t ld,
                              cudaStream_t s);
cudaError_t launch_traj_to_aos(const double *traj, double *aos, uint64_t n_samples, uint64_t n_bodies, uint64_t ld,
                               uint32_t width, cudaStream_t s);
cudaError_t launch_multi_transpose(const MultiColumns &mc, uint64_t n_bodies, uint64_t ld, bool to_soa, cudaStream_t s);
cudaError_t launch_probe_fp64(double *out, int iters, int blocks, cudaStream_t s);
cudaError_t launch_selftest_div(uint64_t seed, uint64_t n_groups, unsigned long long *counts, cudaStream_t s);

} // namespace b200
