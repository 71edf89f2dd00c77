// sm_100a per-body integrator kernels of the six_dof() hot path (K1/K2/K4/K5 of SURVEY §2.4).
//
//   body_exact_kernel       EXACT arithmetic: one thread per body, the whole tick (clear_forces, effectors x4,
//                           calc_accel x4, stage advance x4, final combine, renormalise) in registers, n_ticks
//                           ticks per launch.
//   body_fast_spec_kernel   FAST arithmetic compiled per effector signature (the default FAST route).
//   body_fast_kernel        FAST arithmetic with the run-time effector interpreter (effector lists no signature covers).
//   body_fast_pipe_kernel   opt-in persistent TMA-ring variant of the free-body tick (B200_BODY_CFG=10..14).
#include <algorithm>
#include <cstdint>
#include <cstring>

#include "sixdof_tick.cuh"
#include "sixdof_launch.h"

namespace b200 {

// ================================================================== EXACT body kernel

// SCHED: the launch integrates several ticks of input schedules (P.sched); tick t reads the rows of Tick P.tick_abs + t
template <int INTEG, int BLOCK, int MINB, bool UNR = false, uint32_t SEQ = SEQ_INTERPRET, bool SCHED = false>
__global__ void __launch_bounds__(BLOCK, MINB) body_exact_kernel(const __grid_constant__ StepParams P)
{
    const uint64_t b = (uint64_t)blockIdx.x * BLOCK + threadIdx.x;
    if (b >= P.n_bodies) return;

    Pose x0 = load_pose(P.pos, P.ld, b);
    Motion v0 = load_motion(P.vel, P.ld, b);
    Motion a_out = load_motion(P.acc, P.ld, b);
    Motion f_out = {{0.0, 0.0, 0.0}, {0.0, 0.0, 0.0}};
    const Inertia I = load_inertia(P.ine, P.ld, b);
    const GravReg no_greg{};

    uint32_t traj_phase = 0; // one 64-bit division per launch, not per tick (see fast_ticks)
    uint64_t traj_slot = 0;
    if (P.traj_every) { traj_phase = (uint32_t)(P.tick0 % P.traj_every); traj_slot = P.tick0 / P.traj_every; }
    for (uint32_t t = 0; t < P.n_ticks; ++t) {
        exact_tick<INTEG, false, UNR, SEQ, SCHED>(P, b, x0, v0, a_out, f_out, I, no_greg, P.tick_abs + t);
        if (P.traj_every && ++traj_phase == P.traj_every) {
            traj_phase = 0;
            if (traj_slot < P.traj_capacity) {
                traj_store_state(P, b, traj_slot, x0, v0);
                if (P.traj_planes == 25) traj_store_af(P, b, traj_slot, a_out, f_out);
            }
            ++traj_slot;
        }
    }
    store_pose(P.pos, P.ld, b, x0);
    store_motion(P.vel, P.ld, b, v0);
    store_motion(P.acc, P.ld, b, a_out);
    store_motion(P.frc, P.ld, b, f_out);
}

// ================================================================== FAST body kernels

// Effector columns are consumed inside the (uniform) effector switch, i.e. after the state
// loads and the reciprocal prologue; prefetching them first puts their HBM latency under the
// state loads instead of behind them.
__device__ __forceinline__ void prefetch_effector_columns(const StepParams &P, uint64_t b)
{
    for (uint32_t e = 0; e < P.n_eff; ++e) {
        const double *col = P.eff[e].col;
        if (!col) continue;
        const uint32_t w = P.eff[e].col_width;
        for (uint32_t k = 0; k < w; ++k) asm volatile("prefetch.global.L1 [%0];" ::"l"(col + (uint64_t)k * P.ld + b));
    }
    if (P.gforce)
        for (uint32_t k = 0; k < 9; ++k) asm volatile("prefetch.global.L1 [%0];" ::"l"(P.gforce + (uint64_t)k * P.ld + b));
}

template <int INTEG, int BLOCK, int MINB, bool TRAJ, bool SCHED = false>
__global__ void __launch_bounds__(BLOCK, MINB) body_fast_kernel(const __grid_constant__ StepParams P)
{
    const uint64_t b = (uint64_t)blockIdx.x * BLOCK + threadIdx.x;
    if (b >= P.n_bodies) return;
    prefetch_effector_columns(P, b);
    Pose x0 = load_pose(P.pos, P.ld, b);
    Motion v0 = load_motion(P.vel, P.ld, b);
    const Inertia I = load_inertia(P.ine, P.ld, b);
    Motion a_last, f_last;
    fast_ticks<INTEG, TRAJ, false, SIG_GENERIC, SCHED>(P, b, x0, v0, I, a_last, f_last, P.n_ticks, P.tick0, P.write_fa != 0, GravReg{});
    store_pose(P.pos, P.ld, b, x0);
    store_motion(P.vel, P.ld, b, v0);
    if (P.write_fa) {
        store_motion(P.acc, P.ld, b, a_last);
        store_motion(P.frc, P.ld, b, f_last);
    }
}


// ------------------------------------------------------------------ specialised FAST kernels
//
// One instantiation per (integrator, effector signature): the per-body effector inputs are loaded next to the
// 17 state planes — every load of a body is in flight before the first dependent instruction — and the tick is
// compiled for exactly that effector set.  BPT = bodies per thread: 2 reads every plane as double2 (LDG.E.128,
// body pair 2t, 2t+1) and integrates the pair back to back, so the second body's loads stay in flight under the
// first body's arithmetic.
template <int BPT> struct VecIO;
template <> struct VecIO<1> {
    static __device__ __forceinline__ void ld(const double *p, uint64_t i, double (&o)[1]) { o[0] = p[i]; }
    static __device__ __forceinline__ void st(double *p, uint64_t i, const double (&v)[1], bool) { p[i] = v[0]; }
};
template <> struct VecIO<2> {
    static __device__ __forceinline__ void ld(const double *p, uint64_t i, double (&o)[2])
    {
        const double2 v = *reinterpret_cast<const double2 *>(p + i); // i even, plane base 16-byte aligned (host-checked)
        o[0] = v.x; o[1] = v.y;
    }
    static __device__ __forceinline__ void st(double *p, uint64_t i, const double (&v)[2], bool both)
    {
        if (both) *reinterpret_cast<double2 *>(p + i) = make_double2(v[0], v[1]);
        else p[i] = v[0]; // odd tail: the pair's second body lies outside this launch's range
    }
};

#define B200_LDV(base, plane, expr)                                                        \
    do {                                                                                   \
        double t_[BPT];                                                                    \
        VecIO<BPT>::ld((base) + (uint64_t)(plane) * P.ld, b0, t_);                         \
        _Pragma("unroll") for (int k = 0; k < BPT; ++k) { expr = t_[k]; }                  \
    } while (0)
#define B200_STV(base, plane, expr)                                                        \
    do {                                                                                   \
        double t_[BPT];                                                                    \
        _Pragma("unroll") for (int k = 0; k < BPT; ++k) { t_[k] = expr; }                  \
        VecIO<BPT>::st((base) + (uint64_t)(plane) * P.ld, b0, t_, both);                   \
    } while (0)

// SCHED: the launch integrates several ticks of input schedules (P.sched): the first tick's inputs load with the state
// from the rows of Tick P.tick_abs, every later tick reloads its own rows and refolds (fast_ticks)
template <int INTEG, uint32_t SIG, bool TRAJ, int BLOCK, int MINB, int BPT, bool SCHED = false>
__global__ void __launch_bounds__(BLOCK, MINB) body_fast_spec_kernel(const __grid_constant__ StepParams P)
{
    // Odd launches walk the planes from the far end: the tail of the state the previous launch read and wrote last is
    // still in the 126 MB L2 when this launch starts — read it first, before this launch's own traffic evicts it, and the
    // rewrite lands on lines that are still dirty instead of costing a second DRAM write (scripts/tune_snake.py: 152.4 ->
    // 142.1 us per tick at 2^22 bodies; L2 eviction-class hints on top of it measured nothing and cost registers).
    const unsigned blk = P.reverse ? gridDim.x - 1u - blockIdx.x : blockIdx.x;
    const uint64_t b0 = ((uint64_t)blk * BLOCK + threadIdx.x) * BPT;
    if (b0 >= P.n_bodies) return;
    const bool both = b0 + (BPT - 1) < P.n_bodies;

    Pose x[BPT];
    Motion v[BPT];
    Inertia I[BPT];
    EffIn in[BPT];
    B200_LDV(P.pos, 0, x[k].q.i); B200_LDV(P.pos, 1, x[k].q.j); B200_LDV(P.pos, 2, x[k].q.k); B200_LDV(P.pos, 3, x[k].q.w);
    B200_LDV(P.pos, 4, x[k].x.x); B200_LDV(P.pos, 5, x[k].x.y); B200_LDV(P.pos, 6, x[k].x.z);
    B200_LDV(P.vel, 0, v[k].ang.x); B200_LDV(P.vel, 1, v[k].ang.y); B200_LDV(P.vel, 2, v[k].ang.z);
    B200_LDV(P.vel, 3, v[k].lin.x); B200_LDV(P.vel, 4, v[k].lin.y); B200_LDV(P.vel, 5, v[k].lin.z);
    // the inertia diagonal only matters to invI (a torque) and to the Force column (the launch that writes it back,
    // 25-plane trajectory samples): every other launch leaves its 24 B per body unread.  The mass always matters.
    if (sig_needs_invI(SIG) || P.write_fa || (TRAJ && P.traj_planes == 25)) {
        B200_LDV(P.ine, 0, I[k].diag.x); B200_LDV(P.ine, 1, I[k].diag.y); B200_LDV(P.ine, 2, I[k].diag.z);
    } else {
#pragma unroll
        for (int k = 0; k < BPT; ++k) I[k].diag = Vec3{0.0, 0.0, 0.0};
    }
    B200_LDV(P.ine, 6, I[k].m);
#pragma unroll
    for (int k = 0; k < BPT; ++k) {
        in[k].thrust = 0.0; in[k].cd_rho = in[k].area = 0.0;
        in[k].wr_t = in[k].wr_f = in[k].wind = in[k].wheels = in[k].ww_t = in[k].ww_f = Vec3{0.0, 0.0, 0.0};
    }
    // input columns; a scheduled launch reads the rows of its first tick here
    const double *c_thrust = P.spec.thrust, *c_wr_t = P.spec.wr_t, *c_wr_f = P.spec.wr_f, *c_wheels = P.spec.wheels,
                 *c_wworld = P.spec.wworld, *c_drag = P.spec.drag;
    if constexpr (SCHED) {
        c_thrust = schedule_ptr(c_thrust, P.spec.s_thrust, P.tick_abs);
        c_wr_t = schedule_ptr(c_wr_t, P.spec.s_wrench, P.tick_abs);
        c_wr_f = schedule_ptr(c_wr_f, P.spec.s_wrench, P.tick_abs);
        c_wheels = schedule_ptr(c_wheels, P.spec.s_wheels, P.tick_abs);
        c_wworld = schedule_ptr(c_wworld, P.spec.s_wworld, P.tick_abs);
        c_drag = schedule_ptr(c_drag, P.spec.s_drag, P.tick_abs);
    }
    if (SIG & SIG_THRUST) B200_LDV(c_thrust, 0, in[k].thrust);
    if (SIG & SIG_WRENCH) {
        B200_LDV(c_wr_t, 0, in[k].wr_t.x); B200_LDV(c_wr_t, 1, in[k].wr_t.y); B200_LDV(c_wr_t, 2, in[k].wr_t.z);
        B200_LDV(c_wr_f, 0, in[k].wr_f.x); B200_LDV(c_wr_f, 1, in[k].wr_f.y); B200_LDV(c_wr_f, 2, in[k].wr_f.z);
    }
    if (SIG & SIG_WHEELS) { // the three wheel torques only ever enter as their sum (the rotation is linear)
        Vec3 w[BPT][3];
#pragma unroll
        for (int q = 0; q < 3; ++q) {
            B200_LDV(c_wheels, 3 * q + 0, w[k][q].x); B200_LDV(c_wheels, 3 * q + 1, w[k][q].y); B200_LDV(c_wheels, 3 * q + 2, w[k][q].z);
        }
#pragma unroll
        for (int k = 0; k < BPT; ++k)
            in[k].wheels = Vec3{w[k][0].x + w[k][1].x + w[k][2].x, w[k][0].y + w[k][1].y + w[k][2].y, w[k][0].z + w[k][1].z + w[k][2].z};
    }
    if (SIG & SIG_WWORLD) {
        B200_LDV(c_wworld, 0, in[k].ww_t.x); B200_LDV(c_wworld, 1, in[k].ww_t.y); B200_LDV(c_wworld, 2, in[k].ww_t.z);
        B200_LDV(c_wworld, 3, in[k].ww_f.x); B200_LDV(c_wworld, 4, in[k].ww_f.y); B200_LDV(c_wworld, 5, in[k].ww_f.z);
    }
    if (SIG & SIG_DRAG) {
        B200_LDV(c_drag, 0, in[k].wind.x); B200_LDV(c_drag, 1, in[k].wind.y); B200_LDV(c_drag, 2, in[k].wind.z);
        if (SIG & SIG_DRAG_PB) { B200_LDV(c_drag, 3, in[k].cd_rho); B200_LDV(c_drag, 4, in[k].area); }
    }

    // A (WorldPos, WorldVel) sample on every launch of one tick: the pair stores it from here as one 16-byte store per
    // plane — the per-body 8-byte stores inside fast_ticks fill half of every sector, and the other half arrives a whole
    // tick of arithmetic later (telemetry on every tick: 254 -> see profiles/r02_tune_telemetry.txt)
    const bool defer_traj = TRAJ && BPT == 2 && both && P.n_ticks == 1 && P.traj_planes == 13;
    Motion a_last[BPT], f_last[BPT];
    // Force-free tick: every stage acceleration is (0*m)*rcp(m), +-0 for a finite nonzero mass, so the new velocity has
    // the loaded bits except for a -0 component, a degenerate mass (NaN) or a NaN payload.  Bit j of vdirty: velocity
    // plane j changed for a body of this thread (compared as integers: +-0 and NaN payloads count).  Planes that did
    // not change are not stored, and their L2 lines stay clean instead of costing a DRAM write-back.  The pair's
    // second body outside the range (odd tail) is not integrated, so it never marks a plane.
    uint32_t vdirty = 0x3fu;
#pragma unroll
    for (int k = 0; k < BPT; ++k) {
        const Motion v_in = v[k];
        if (k == 0 || both)
            fast_ticks<INTEG, TRAJ, false, SIG, SCHED>(P, b0 + k, x[k], v[k], I[k], a_last[k], f_last[k], P.n_ticks, P.tick0,
                                                       P.write_fa != 0, GravReg{}, in[k], !defer_traj);
        if (SIG == SIG_FREE) {
            if (k == 0) vdirty = 0u;
            auto ne = [](double a, double b) { return (uint32_t)(__double_as_longlong(a) != __double_as_longlong(b)); };
            vdirty |= ne(v_in.ang.x, v[k].ang.x) | ne(v_in.ang.y, v[k].ang.y) << 1 | ne(v_in.ang.z, v[k].ang.z) << 2 |
                      ne(v_in.lin.x, v[k].lin.x) << 3 | ne(v_in.lin.y, v[k].lin.y) << 4 | ne(v_in.lin.z, v[k].lin.z) << 5;
        }
    }
    if (TRAJ && BPT == 2 && defer_traj && P.traj_every) {
        const uint64_t after = P.tick0 + 1;
        const uint64_t slot = after / P.traj_every - 1;
        if (after % P.traj_every == 0 && slot < P.traj_capacity) {
            double *t = P.traj + slot * 13ull * P.ld + b0;
            auto put = [&](int plane, double v0, double v1) { __stcs(reinterpret_cast<double2 *>(t + (uint64_t)plane * P.ld), make_double2(v0, v1)); };
            constexpr int o = BPT - 1; // index of the pair's second body (0 when the kernel is compiled for one body per thread)
            put(0, x[0].q.i, x[o].q.i); put(1, x[0].q.j, x[o].q.j); put(2, x[0].q.k, x[o].q.k); put(3, x[0].q.w, x[o].q.w);
            put(4, x[0].x.x, x[o].x.x); put(5, x[0].x.y, x[o].x.y); put(6, x[0].x.z, x[o].x.z);
            put(7, v[0].ang.x, v[o].ang.x); put(8, v[0].ang.y, v[o].ang.y); put(9, v[0].ang.z, v[o].ang.z);
            put(10, v[0].lin.x, v[o].lin.x); put(11, v[0].lin.y, v[o].lin.y); put(12, v[0].lin.z, v[o].lin.z);
        }
    }

    B200_STV(P.pos, 0, x[k].q.i); B200_STV(P.pos, 1, x[k].q.j); B200_STV(P.pos, 2, x[k].q.k); B200_STV(P.pos, 3, x[k].q.w);
    B200_STV(P.pos, 4, x[k].x.x); B200_STV(P.pos, 5, x[k].x.y); B200_STV(P.pos, 6, x[k].x.z);
    if (vdirty & 1u) B200_STV(P.vel, 0, v[k].ang.x);
    if (vdirty & 2u) B200_STV(P.vel, 1, v[k].ang.y);
    if (vdirty & 4u) B200_STV(P.vel, 2, v[k].ang.z);
    if (vdirty & 8u) B200_STV(P.vel, 3, v[k].lin.x);
    if (vdirty & 16u) B200_STV(P.vel, 4, v[k].lin.y);
    if (vdirty & 32u) B200_STV(P.vel, 5, v[k].lin.z);
    if (P.write_fa) {
        B200_STV(P.acc, 0, a_last[k].ang.x); B200_STV(P.acc, 1, a_last[k].ang.y); B200_STV(P.acc, 2, a_last[k].ang.z);
        B200_STV(P.acc, 3, a_last[k].lin.x); B200_STV(P.acc, 4, a_last[k].lin.y); B200_STV(P.acc, 5, a_last[k].lin.z);
        B200_STV(P.frc, 0, f_last[k].ang.x); B200_STV(P.frc, 1, f_last[k].ang.y); B200_STV(P.frc, 2, f_last[k].ang.z);
        B200_STV(P.frc, 3, f_last[k].lin.x); B200_STV(P.frc, 4, f_last[k].lin.y); B200_STV(P.frc, 5, f_last[k].lin.z);
    }
}

// ------------------------------------------------------------------ TMA-pipelined persistent variant
//
// One CTA = kPipeTB threads = one tile of kPipeTB bodies at a time, looping over tiles
// (persistent grid sized to the SM count).  The 17 input planes of the next tiles
// (pos 7, vel 6, inertia diag 3 + mass) are fetched with cp.async.bulk into a
// kStages-deep shared-memory ring, completion signalled on mbarriers; the 13 output
// planes leave through a double-buffered shared-memory tile and cp.async.bulk stores.
// The FP64 work of tile i therefore overlaps the HBM traffic of tiles i+1.. and i-1,
// which the direct kernel (1 CTA/SM at 150+ registers) cannot do.
static constexpr int kPipeTB = 128;
static constexpr int kPipeIn = 17;
static constexpr int kPipeOut = 13;

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *dst_smem, const void *src_gmem, uint32_t bytes, uint64_t *bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void bulk_s2g(void *dst_gmem, const void *src_smem, uint32_t bytes)
{
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst_gmem), "r"(smem_u32(src_smem)),
                 "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// DIRECT_OUT: results leave with plain coalesced stores (no output tiles), which shrinks the CTA to
// STAGES x 17 KB of shared memory so that 4 CTAs/SM fit at 128 registers — the input ring then keeps
// ~17 KB per CTA in flight at all times, independent of how long the FP64 phase of a tile takes.
template <int INTEG, int STAGES, int MINB, bool DIRECT_OUT>
__global__ void __launch_bounds__(kPipeTB, MINB) body_fast_pipe_kernel(const __grid_constant__ StepParams P)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    constexpr int kOutTiles = DIRECT_OUT ? 0 : 2;
    double(*sin)[kPipeIn][kPipeTB] = reinterpret_cast<double(*)[kPipeIn][kPipeTB]>(smem_raw);
    double(*sout)[kPipeOut][kPipeTB] =
        reinterpret_cast<double(*)[kPipeOut][kPipeTB]>(smem_raw + sizeof(double) * STAGES * kPipeIn * kPipeTB);
    uint64_t *full = reinterpret_cast<uint64_t *>(smem_raw + sizeof(double) * (STAGES * kPipeIn + kOutTiles * kPipeOut) * kPipeTB);

    const int tid = threadIdx.x;
    const uint64_t n_tiles = (P.n_bodies + kPipeTB - 1) / kPipeTB;
    constexpr uint32_t kPlaneBytes = kPipeTB * sizeof(double);

    if (tid == 0) {
        for (int s = 0; s < STAGES; ++s) mbar_init(&full[s], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    // source plane of input slot k for the tile starting at body b0
    auto src_plane = [&](int k, uint64_t b0) -> const double * {
        if (k < 7) return P.pos + (uint64_t)k * P.ld + b0;
        if (k < 13) return P.vel + (uint64_t)(k - 7) * P.ld + b0;
        return P.ine + (uint64_t)(k == 16 ? 6 : k - 13) * P.ld + b0;
    };
    auto issue_loads = [&](uint64_t tile, int s) { // warp 0
        if (tid == 0) mbar_expect_tx(&full[s], kPipeIn * kPlaneBytes);
        __syncwarp();
        if (tid < kPipeIn) bulk_g2s(&sin[s][tid][0], src_plane(tid, tile * kPipeTB), kPlaneBytes, &full[s]);
    };

    if (tid < 32)
        for (int s = 0; s < STAGES; ++s) {
            const uint64_t tile = blockIdx.x + (uint64_t)s * gridDim.x;
            if (tile < n_tiles) issue_loads(tile, s);
        }

    uint32_t it = 0;
    for (uint64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++it) {
        const int s = it % STAGES;
        const uint32_t parity = (it / STAGES) & 1u;
        const uint64_t b = tile * kPipeTB + tid;
        mbar_wait(&full[s], parity);
        Pose x0;
        Motion v0;
        Inertia I;
        x0.q = Quat{sin[s][0][tid], sin[s][1][tid], sin[s][2][tid], sin[s][3][tid]};
        x0.x = Vec3{sin[s][4][tid], sin[s][5][tid], sin[s][6][tid]};
        v0.ang = Vec3{sin[s][7][tid], sin[s][8][tid], sin[s][9][tid]};
        v0.lin = Vec3{sin[s][10][tid], sin[s][11][tid], sin[s][12][tid]};
        I.diag = Vec3{sin[s][13][tid], sin[s][14][tid], sin[s][15][tid]};
        I.m = sin[s][16][tid];
        // the output tile about to be written was handed to the async proxy two tiles ago
        if (!DIRECT_OUT && tid < kPipeOut) bulk_wait_read<1>();
        __syncthreads(); // everyone has drained stage s; out[it&1] is free
        if (tid < 32) {
            const uint64_t next = tile + (uint64_t)STAGES * gridDim.x;
            if (next < n_tiles) issue_loads(next, s);
        }
        Motion a_last, f_last;
        const bool live = b < P.n_bodies;
        if (live) fast_ticks<INTEG, true>(P, b, x0, v0, I, a_last, f_last, P.n_ticks, P.tick0, P.write_fa != 0, GravReg{});
        if (DIRECT_OUT) {
            if (live) {
                store_pose(P.pos, P.ld, b, x0);
                store_motion(P.vel, P.ld, b, v0);
                if (P.write_fa) {
                    store_motion(P.acc, P.ld, b, a_last);
                    store_motion(P.frc, P.ld, b, f_last);
                }
            }
            continue;
        }
        const int ob = it & 1;
        sout[ob][0][tid] = x0.q.i; sout[ob][1][tid] = x0.q.j; sout[ob][2][tid] = x0.q.k; sout[ob][3][tid] = x0.q.w;
        sout[ob][4][tid] = x0.x.x; sout[ob][5][tid] = x0.x.y; sout[ob][6][tid] = x0.x.z;
        sout[ob][7][tid] = v0.ang.x; sout[ob][8][tid] = v0.ang.y; sout[ob][9][tid] = v0.ang.z;
        sout[ob][10][tid] = v0.lin.x; sout[ob][11][tid] = v0.lin.y; sout[ob][12][tid] = v0.lin.z;
        if (live && P.write_fa) {
            store_motion(P.acc, P.ld, b, a_last);
            store_motion(P.frc, P.ld, b, f_last);
        }
        fence_async_smem();
        __syncthreads();
        if (tid < kPipeOut) {
            double *dst = (tid < 7 ? P.pos + (uint64_t)tid * P.ld : P.vel + (uint64_t)(tid - 7) * P.ld) + tile * kPipeTB;
            bulk_s2g(dst, &sout[ob][tid][0], kPlaneBytes);
            bulk_commit();
        }
    }
    if (!DIRECT_OUT && tid < kPipeOut) bulk_wait_all();
}

// ================================================================== launchers

// the instantiation without trajectory code for launches that record nothing, the generic one otherwise
#define BODY_FAST(INTEG, BLOCK, MINB)                                                        \
    do {                                                                                     \
        if (P.traj_every) body_fast_kernel<INTEG, BLOCK, MINB, true><<<g(BLOCK), BLOCK, 0, s>>>(P);  \
        else body_fast_kernel<INTEG, BLOCK, MINB, false><<<g(BLOCK), BLOCK, 0, s>>>(P);      \
    } while (0)

// ------------------------------------------------------------------ effector list -> signature
//
// A signature covers an effector list when the folded result does not depend on anything the compile-time form
// cannot express: no entity masks (query-join membership), at most one thrust / wrench / drag / frame effector,
// no wrench ahead of the drag (apply_drag resets the torque accumulated before it), a drag that has its wind
// column, the edge_fold gravity first.  Everything else keeps the run-time interpreter.  A list that applies no force
// at all (empty, or constant gravities that sum to exactly zero) is SIG_FREE.
static uint32_t spec_signature(StepParams &Q)
{
    uint32_t sig = 0;
    int n_thrust = 0, n_wrench = 0, n_drag = 0, n_frame = 0;
    bool wrench_seen = false;
    StepParams::Spec sp{};
    for (uint32_t i = 0; i < Q.n_eff; ++i) {
        const EffDev &E = Q.eff[i];
        if (E.mask) return SIG_GENERIC;
        switch (E.kind) {
        case B200_EFF_GRAVITY_CONST:
            sp.g[0] += E.p[0]; sp.g[1] += E.p[1]; sp.g[2] += E.p[2];
            break;
        case B200_EFF_DRAG_QUADRATIC:
            if (!E.col || wrench_seen || ++n_drag > 1) return SIG_GENERIC;
            sig |= SIG_DRAG | (E.col_width == 5 ? SIG_DRAG_PB : 0u);
            sp.kd = 0.5 * E.p[0] * E.p[1];
            sp.drag = E.col;
            sp.s_drag = E.sched;
            break;
        case B200_EFF_THRUST_BODY:
            if (!E.col || ++n_thrust > 1) return SIG_GENERIC;
            sig |= SIG_THRUST;
            sp.axis[0] = E.p[0]; sp.axis[1] = E.p[1]; sp.axis[2] = E.p[2];
            sp.thrust = E.col;
            sp.s_thrust = E.sched;
            break;
        case B200_EFF_WRENCH_BODY: {
            if (!E.col || ++n_wrench > 1) return SIG_GENERIC;
            wrench_seen = true;
            sig |= SIG_WRENCH;
            const uint64_t to = (E.flags & B200_EFF_FLAG_WRENCH_LINEAR_FIRST) ? 3 : 0;
            sp.wr_t = E.col + to * Q.ld;
            sp.wr_f = E.col + (3 - to) * Q.ld;
            sp.s_wrench = E.sched;
            break;
        }
        case B200_EFF_GRAVITY_FRAME:
            if (++n_frame > 1) return SIG_GENERIC;
            sig |= SIG_FRAME;
            sp.mu = E.p[0]; sp.om[0] = E.p[1]; sp.om[1] = E.p[2]; sp.om[2] = E.p[3];
            break;
        case B200_EFF_GRAVITY_EDGES_NEWTON:
        case B200_EFF_GRAVITY_EDGES_SOFTENED:
            if (i != 0 || !Q.gforce || !Q.has_edge) return SIG_GENERIC;
            sig |= SIG_GRAPH;
            break;
        case B200_EFF_GRAVITY_J2:
            if (sig & SIG_J2) return SIG_GENERIC;
            sig |= SIG_J2;
            sp.j2_mu = E.p[0]; sp.j2_k = E.p[1] * E.p[2] * E.p[2];
            break;
        case B200_EFF_WRENCH_WORLD:
            if (!E.col || (sig & SIG_WWORLD)) return SIG_GENERIC;
            sig |= SIG_WWORLD;
            sp.wworld = E.col;
            sp.s_wworld = E.sched;
            break;
        case B200_EFF_TORQUE_BODY_FOLD: // the fold overwrites Force: only as the first effector is it a plain torque term
            if (i != 0 || !E.col || E.col_width != 9) return SIG_GENERIC;
            sig |= SIG_WHEELS;
            sp.wheels = E.col;
            sp.s_wheels = E.sched;
            break;
        default: return SIG_GENERIC;
        }
    }
    Q.spec = sp;
    if (sig == 0u && sp.g[0] == 0.0 && sp.g[1] == 0.0 && sp.g[2] == 0.0) return SIG_FREE;
    return sig;
}

// launch shape of the specialised kernels: (threads per CTA, resident CTAs per SM the register allocation is bounded
// for, bodies per thread).  B200_SPEC_CFG selects among the shapes a tuning build (-DB200_TUNE) instantiates.
template <int INTEG, uint32_t SIG, bool TRAJ, int BLOCK, int MINB, int BPT, bool SCHED = false>
static void launch_spec_shape(const StepParams &Q, cudaStream_t s)
{
    const uint64_t threads = (Q.n_bodies + BPT - 1) / BPT;
    const unsigned grid = (unsigned)((threads + BLOCK - 1) / BLOCK);
    body_fast_spec_kernel<INTEG, SIG, TRAJ, BLOCK, MINB, BPT, SCHED><<<grid, BLOCK, 0, s>>>(Q);
}

static bool planes_16B_aligned(const StepParams &Q, uint32_t sig)
{
    uintptr_t a = (uintptr_t)Q.pos | (uintptr_t)Q.vel | (uintptr_t)Q.ine | (uintptr_t)Q.acc | (uintptr_t)Q.frc | (uintptr_t)Q.traj;
    if (sig & SIG_THRUST) a |= (uintptr_t)Q.spec.thrust;
    if (sig & SIG_WRENCH) a |= (uintptr_t)Q.spec.wr_t | (uintptr_t)Q.spec.wr_f;
    if (sig & SIG_DRAG) a |= (uintptr_t)Q.spec.drag;
    if (sig & SIG_WHEELS) a |= (uintptr_t)Q.spec.wheels;
    if (sig & SIG_WWORLD) a |= (uintptr_t)Q.spec.wworld;
    // every row of a scheduled column starts a whole number of rows (width * ld doubles) after the table base
    const uint64_t strides = Q.spec.s_thrust.stride | Q.spec.s_wrench.stride | Q.spec.s_drag.stride | Q.spec.s_wheels.stride |
                             Q.spec.s_wworld.stride;
    return (a & 15u) == 0 && (Q.ld & 1u) == 0 && (strides & 1u) == 0;
}

// Default shape, measured on B200 at 2^22 worlds (profiles/r02_tune_spec.md): body pairs (BPT = 2, LDG.E.128) at
// 128 threads x 3 CTAs/SM (<= 168 registers, no spills) run the free / rocket / falcon9 signatures at 7.2 TB/s of
// algorithmic bytes; one body per thread at 128 x 4 is 9 % (rocket) to 11 % (falcon9) slower.  Ranges too small to
// fill the machine with pairs, or whose planes are not 16-byte aligned (odd world-range offsets), take one body
// per thread.
template <int INTEG, uint32_t SIG, bool TRAJ, bool SCHED = false>
static void launch_spec(const StepParams &Q, cudaStream_t s)
{
    const bool vec_ok = planes_16B_aligned(Q, SIG);
    if constexpr (SCHED) { // the default shapes only
        constexpr uint64_t kPairMinBodies = 2ull * 128 * 3 * 148;
        if (vec_ok && Q.n_bodies >= kPairMinBodies) launch_spec_shape<INTEG, SIG, TRAJ, 128, 3, 2, true>(Q, s);
        else launch_spec_shape<INTEG, SIG, TRAJ, 128, 4, 1, true>(Q, s);
        return;
    }
#ifdef B200_TUNE
    const int cfg = env_int("B200_SPEC_CFG", -1); // re-read per launch: one tuning process sweeps the shapes
    switch (cfg) {
    case 0: launch_spec_shape<INTEG, SIG, TRAJ, 128, 4, 1>(Q, s); return;
    case 1: launch_spec_shape<INTEG, SIG, TRAJ, 128, 5, 1>(Q, s); return;
    case 2: launch_spec_shape<INTEG, SIG, TRAJ, 128, 6, 1>(Q, s); return;
    case 3: launch_spec_shape<INTEG, SIG, TRAJ, 256, 2, 1>(Q, s); return;
    case 4: if (vec_ok) { launch_spec_shape<INTEG, SIG, TRAJ, 128, 3, 2>(Q, s); return; } break;
    case 5: if (vec_ok) { launch_spec_shape<INTEG, SIG, TRAJ, 128, 4, 2>(Q, s); return; } break;
    case 6: if (vec_ok) { launch_spec_shape<INTEG, SIG, TRAJ, 128, 2, 2>(Q, s); return; } break;
    case 7: if (vec_ok) { launch_spec_shape<INTEG, SIG, TRAJ, 64, 6, 2>(Q, s); return; } break;
    case 8: launch_spec_shape<INTEG, SIG, TRAJ, 64, 10, 1>(Q, s); return;
    default: break;
    }
#endif
    constexpr uint64_t kPairMinBodies = 2ull * 128 * 3 * 148; // one full wave of body pairs
    if (vec_ok && Q.n_bodies >= kPairMinBodies) launch_spec_shape<INTEG, SIG, TRAJ, 128, 3, 2>(Q, s);
    else launch_spec_shape<INTEG, SIG, TRAJ, 128, 4, 1>(Q, s);
}

// signatures with a compiled kernel; anything else falls back to the interpreter kernel
#ifdef B200_TUNE
#define B200_SPEC_SIGS(X) X(SIG_FREE) X(0u) X(SIG_THRUST | SIG_DRAG) X(SIG_FRAME | SIG_WRENCH)
#else
#define B200_SPEC_SIGS(X)                                                                                        \
    X(SIG_FREE) X(0u) X(SIG_DRAG) X(SIG_THRUST) X(SIG_WRENCH) X(SIG_FRAME) X(SIG_GRAPH)                                       \
    X(SIG_THRUST | SIG_DRAG) X(SIG_THRUST | SIG_DRAG | SIG_DRAG_PB) X(SIG_THRUST | SIG_WRENCH) X(SIG_FRAME | SIG_WRENCH)     \
    X(SIG_J2) X(SIG_WHEELS | SIG_J2) X(SIG_WWORLD) X(SIG_WHEELS | SIG_WWORLD)
#endif

// the signatures that read an input column, compiled a second time for fused launches with input schedules
#ifdef B200_TUNE
#define B200_SCHED_SIGS(X) X(SIG_THRUST | SIG_DRAG)
#else
#define B200_SCHED_SIGS(X)                                                                                                 \
    X(SIG_DRAG) X(SIG_THRUST) X(SIG_WRENCH) X(SIG_THRUST | SIG_DRAG) X(SIG_THRUST | SIG_DRAG | SIG_DRAG_PB)                \
    X(SIG_THRUST | SIG_WRENCH) X(SIG_FRAME | SIG_WRENCH) X(SIG_WHEELS | SIG_J2) X(SIG_WWORLD) X(SIG_WHEELS | SIG_WWORLD)
#endif

template <int INTEG>
static bool launch_spec_sig(const StepParams &Q, uint32_t sig, cudaStream_t s)
{
    const bool traj = Q.traj_every != 0;
    if (Q.sched) {
        switch (sig) {
#define X(SIGV)                                                                \
    case (SIGV):                                                               \
        if (traj) launch_spec<INTEG, (SIGV), true, true>(Q, s);                \
        else launch_spec<INTEG, (SIGV), false, true>(Q, s);                    \
        return true;
            B200_SCHED_SIGS(X)
#undef X
        default: return false;
        }
    }
    switch (sig) {
#define X(SIGV)                                                                \
    case (SIGV):                                                               \
        if (traj) launch_spec<INTEG, (SIGV), true>(Q, s);                      \
        else launch_spec<INTEG, (SIGV), false>(Q, s);                          \
        return true;
        B200_SPEC_SIGS(X)
#undef X
    default: return false;
    }
}

// EXACT effector sequences with a compiled kernel (four bits per effector kind, list order); every other list —
// and any list with an entity mask — runs the interpreter kernel
#define B200_SEQ1(a) ((uint32_t)(a))
#define B200_SEQ2(a, b) ((uint32_t)(a) | ((uint32_t)(b) << 4))
#define B200_SEQ3(a, b, c) ((uint32_t)(a) | ((uint32_t)(b) << 4) | ((uint32_t)(c) << 8))
#define B200_EXACT_SEQS(X)                                                                                              \
    X(0u)                                                                                                               \
    X(B200_SEQ1(B200_EFF_GRAVITY_CONST))                                                                                \
    X(B200_SEQ2(B200_EFF_GRAVITY_CONST, B200_EFF_DRAG_QUADRATIC))                            /* ball/sim.py */          \
    X(B200_SEQ3(B200_EFF_GRAVITY_CONST, B200_EFF_THRUST_BODY, B200_EFF_DRAG_QUADRATIC))      /* rocket Monte-Carlo */   \
    X(B200_SEQ3(B200_EFF_GRAVITY_CONST, B200_EFF_THRUST_BODY, B200_EFF_WRENCH_BODY))         /* rocket/main.py */       \
    X(B200_SEQ2(B200_EFF_GRAVITY_FRAME, B200_EFF_WRENCH_BODY))                               /* falcon9/sim.py */       \
    X(B200_SEQ1(B200_EFF_GRAVITY_EDGES_NEWTON)) X(B200_SEQ1(B200_EFF_GRAVITY_EDGES_SOFTENED))                         \
    X(B200_SEQ2(B200_EFF_TORQUE_BODY_FOLD, B200_EFF_WRENCH_WORLD))                           /* cube-sat replay */

static uint32_t exact_sequence(const StepParams &P)
{
    if (P.n_eff > 5) return SEQ_INTERPRET;
    uint32_t seq = 0;
    for (uint32_t i = 0; i < P.n_eff; ++i) {
        if (P.eff[i].mask || P.eff[i].kind == 0 || P.eff[i].kind > 15) return SEQ_INTERPRET;
        seq |= P.eff[i].kind << (4 * i);
    }
    return seq;
}

// the sequences that read an input column, compiled a second time for fused launches with input schedules
#define B200_EXACT_SCHED_SEQS(X)                                                                                        \
    X(B200_SEQ2(B200_EFF_GRAVITY_CONST, B200_EFF_DRAG_QUADRATIC))                                                       \
    X(B200_SEQ3(B200_EFF_GRAVITY_CONST, B200_EFF_THRUST_BODY, B200_EFF_DRAG_QUADRATIC))                                 \
    X(B200_SEQ3(B200_EFF_GRAVITY_CONST, B200_EFF_THRUST_BODY, B200_EFF_WRENCH_BODY))                                    \
    X(B200_SEQ2(B200_EFF_GRAVITY_FRAME, B200_EFF_WRENCH_BODY))                                                          \
    X(B200_SEQ2(B200_EFF_TORQUE_BODY_FOLD, B200_EFF_WRENCH_WORLD))

template <int INTEG, int BLOCK, int MINB>
static bool launch_exact_sched(const StepParams &P, uint32_t seq, cudaStream_t s)
{
    const unsigned grid = (unsigned)((P.n_bodies + BLOCK - 1) / BLOCK);
    switch (seq) {
#define X(SEQV)                                                                            \
    case (SEQV):                                                                           \
        body_exact_kernel<INTEG, BLOCK, MINB, false, (SEQV), true><<<grid, BLOCK, 0, s>>>(P); \
        return true;
        B200_EXACT_SCHED_SEQS(X)
#undef X
    default: body_exact_kernel<INTEG, BLOCK, MINB, false, SEQ_INTERPRET, true><<<grid, BLOCK, 0, s>>>(P); return true;
    }
}

template <int INTEG, int BLOCK, int MINB>
static bool launch_exact_seq(const StepParams &P, uint32_t seq, cudaStream_t s)
{
    const unsigned grid = (unsigned)((P.n_bodies + BLOCK - 1) / BLOCK);
    switch (seq) {
#define X(SEQV)                                                                            \
    case (SEQV):                                                                           \
        body_exact_kernel<INTEG, BLOCK, MINB, false, (SEQV)><<<grid, BLOCK, 0, s>>>(P);    \
        return true;
        B200_EXACT_SEQS(X)
#undef X
    default: return false;
    }
}

cudaError_t launch_body_step(const StepParams &P, int integrator, int math_mode, cudaStream_t s)
{
    if (P.n_bodies == 0) return cudaSuccess;
    const bool rk4 = integrator == B200_INTEGRATOR_RK4;
    if (P.sched) {
        // several ticks of input schedules in one launch: the kernels compiled to read each tick's rows, in the default
        // shapes (the tuning switches below do not apply)
        if (math_mode == B200_MATH_EXACT) {
            const uint32_t seq = exact_sequence(P);
            if (rk4) launch_exact_sched<B200_INTEGRATOR_RK4, 128, 4>(P, seq, s);
            else launch_exact_sched<B200_INTEGRATOR_SEMI_IMPLICIT, 256, 1>(P, seq, s);
            return cudaGetLastError();
        }
        StepParams Q = P;
        const uint32_t sig = spec_signature(Q);
        const bool done = sig != SIG_GENERIC && (rk4 ? launch_spec_sig<B200_INTEGRATOR_RK4>(Q, sig, s)
                                                     : launch_spec_sig<B200_INTEGRATOR_SEMI_IMPLICIT>(Q, sig, s));
        if (!done) {
            auto g = [&](int blk) { return (unsigned)((P.n_bodies + blk - 1) / blk); };
            if (rk4) {
                if (P.traj_every) body_fast_kernel<B200_INTEGRATOR_RK4, 128, 4, true, true><<<g(128), 128, 0, s>>>(P);
                else body_fast_kernel<B200_INTEGRATOR_RK4, 128, 4, false, true><<<g(128), 128, 0, s>>>(P);
            } else {
                if (P.traj_every) body_fast_kernel<B200_INTEGRATOR_SEMI_IMPLICIT, 128, 4, true, true><<<g(128), 128, 0, s>>>(P);
                else body_fast_kernel<B200_INTEGRATOR_SEMI_IMPLICIT, 128, 4, false, true><<<g(128), 128, 0, s>>>(P);
            }
        }
        return cudaGetLastError();
    }
    if (math_mode == B200_MATH_EXACT) {
#ifdef B200_TUNE
        const int xcfg = env_int("B200_EXACT_CFG", 3);
#else
        static const int xcfg = env_int("B200_EXACT_CFG", 3);
#endif
        auto g = [&](int blk) { return (unsigned)((P.n_bodies + blk - 1) / blk); };
        // default: the kernel compiled for this effector sequence (no interpreter: 5.4e9 vs 4.1e9 entity-steps/s on free
        // bodies, profiles/r02_tune_misc.md); the interpreter kernel for every other list
        if (xcfg == 3) {
            const uint32_t seq = exact_sequence(P);
#ifdef B200_TUNE
            if (seq != SEQ_INTERPRET && rk4) switch (env_int("B200_EXACT_SEQ_CFG", 0)) { // registers vs warps for the compiled sequences
            case 1: if (launch_exact_seq<B200_INTEGRATOR_RK4, 128, 3>(P, seq, s)) return cudaGetLastError(); break;
            case 2: if (launch_exact_seq<B200_INTEGRATOR_RK4, 128, 2>(P, seq, s)) return cudaGetLastError(); break;
            case 3: if (launch_exact_seq<B200_INTEGRATOR_RK4, 64, 6>(P, seq, s)) return cudaGetLastError(); break;
            case 4: if (launch_exact_seq<B200_INTEGRATOR_RK4, 128, 5>(P, seq, s)) return cudaGetLastError(); break;
            default: break;
            }
#endif
            if (seq != SEQ_INTERPRET &&
                (rk4 ? launch_exact_seq<B200_INTEGRATOR_RK4, 128, 4>(P, seq, s) : launch_exact_seq<B200_INTEGRATOR_SEMI_IMPLICIT, 256, 1>(P, seq, s)))
                return cudaGetLastError();
        }
        if (!rk4) body_exact_kernel<B200_INTEGRATOR_SEMI_IMPLICIT, 256, 1><<<g(256), 256, 0, s>>>(P);
        else switch (xcfg) {
        case 1: body_exact_kernel<B200_INTEGRATOR_RK4, 256, 2><<<g(256), 256, 0, s>>>(P); break;
        case 0: body_exact_kernel<B200_INTEGRATOR_RK4, 256, 1><<<g(256), 256, 0, s>>>(P); break;
#ifdef B200_TUNE
        case 4: body_exact_kernel<B200_INTEGRATOR_RK4, 128, 5><<<g(128), 128, 0, s>>>(P); break;
        case 5: body_exact_kernel<B200_INTEGRATOR_RK4, 128, 6><<<g(128), 128, 0, s>>>(P); break;
        case 6: body_exact_kernel<B200_INTEGRATOR_RK4, 64, 12><<<g(64), 64, 0, s>>>(P); break;
        case 7: body_exact_kernel<B200_INTEGRATOR_RK4, 128, 3, true><<<g(128), 128, 0, s>>>(P); break;
        case 8: body_exact_kernel<B200_INTEGRATOR_RK4, 128, 2, true><<<g(128), 128, 0, s>>>(P); break;
        case 9: body_exact_kernel<B200_INTEGRATOR_RK4, 128, 4, true><<<g(128), 128, 0, s>>>(P); break;
        case 10: body_exact_kernel<B200_INTEGRATOR_RK4, 128, 3, true, 0u><<<g(128), 128, 0, s>>>(P); break;
        case 11: body_exact_kernel<B200_INTEGRATOR_RK4, 128, 5, false, 0u><<<g(128), 128, 0, s>>>(P); break;
#endif
        default: body_exact_kernel<B200_INTEGRATOR_RK4, 128, 4><<<g(128), 128, 0, s>>>(P); break; // 12: interpreter kept
        }
        return cudaGetLastError();
    }
    static const int cfg = env_int("B200_BODY_CFG", 3);
    auto g = [&](int blk) { return (unsigned)((P.n_bodies + blk - 1) / blk); };
    if (cfg >= 10 && cfg <= 14 && rk4) {
        // opt-in persistent TMA-pipelined kernel: whole 128-body tiles, so the range must start on a tile boundary
        // of 16-byte aligned planes and hold whole tiles; any other range runs the default kernels below
        const bool tiles_ok = ((uintptr_t)P.pos % 1024u) == 0 && ((uintptr_t)P.vel % 1024u) == 0 && ((uintptr_t)P.ine % 1024u) == 0 &&
                              P.ld % kPipeTB == 0 && P.n_bodies % kPipeTB == 0;
        if (tiles_ok) {
            const bool direct = cfg >= 13;
            const int stages = cfg == 10 ? 2 : (cfg == 11 ? 3 : (cfg == 12 ? 4 : (cfg == 13 ? 2 : 3)));
            const size_t smem = sizeof(double) * (stages * kPipeIn + (direct ? 0 : 2) * kPipeOut) * kPipeTB + 8 * stages;
            auto kern = cfg == 10 ? body_fast_pipe_kernel<B200_INTEGRATOR_RK4, 2, 3, false>
                      : cfg == 11 ? body_fast_pipe_kernel<B200_INTEGRATOR_RK4, 3, 2, false>
                      : cfg == 12 ? body_fast_pipe_kernel<B200_INTEGRATOR_RK4, 4, 2, false>
                      : cfg == 13 ? body_fast_pipe_kernel<B200_INTEGRATOR_RK4, 2, 4, true>
                                  : body_fast_pipe_kernel<B200_INTEGRATOR_RK4, 3, 4, true>;
            // opt-in tuning variant: attributes are (re)set on every launch, cheap next to a >100 us kernel
            int dev = 0, sm_count = 0, per_sm = 0;
            cudaGetDevice(&dev);
            cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, dev);
            cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kPipeTB, smem);
            if (per_sm < 1) per_sm = 1;
            const uint64_t n_tiles = P.n_bodies / kPipeTB;
            const unsigned grid_p = (unsigned)std::min<uint64_t>(n_tiles, (uint64_t)sm_count * per_sm);
            kern<<<grid_p, kPipeTB, smem, s>>>(P);
            return cudaGetLastError();
        }
    }
    // default: the kernel compiled for this effector signature; the interpreter kernel for the lists none covers
#ifdef B200_TUNE
    const int no_spec = env_int("B200_NO_SPEC", 0);
#else
    static const int no_spec = env_int("B200_NO_SPEC", 0);
#endif
    StepParams Q = P;
    static const int snake = env_int("B200_SNAKE", 1);
    if (!snake) Q.reverse = 0; // A/B switch: always walk forward
    const uint32_t sig = no_spec ? (uint32_t)SIG_GENERIC : spec_signature(Q);
    bool done = false;
    if (sig != SIG_GENERIC) done = rk4 ? launch_spec_sig<B200_INTEGRATOR_RK4>(Q, sig, s)
                                       : launch_spec_sig<B200_INTEGRATOR_SEMI_IMPLICIT>(Q, sig, s);
    if (!done) {
        // 128 threads x 4 CTAs/SM = 16 warps/SM at <= 128 registers (profiles/r01_tuning.md)
        if (rk4) BODY_FAST(B200_INTEGRATOR_RK4, 128, 4);
        else BODY_FAST(B200_INTEGRATOR_SEMI_IMPLICIT, 128, 4);
    }
    return cudaGetLastError();
}

} // namespace b200
