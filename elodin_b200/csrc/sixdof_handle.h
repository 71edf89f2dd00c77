// Internals of a b200_sixdof handle, shared by the translation units that implement the C ABI
// (sixdof_abi.cu: executor; sixdof_comm.cu: NCCL gather, peer-memory row sharding).
#pragma once
#include <cstdarg>
#include <cstdio>
#include <string>
#include <vector>

#include "sixdof_internal.h"

namespace b200 {

int fail(int code, const char *fmt, ...);          // sets the thread-local message, returns code
const char *last_error_message();

struct Column {
    uint64_t id;
    uint32_t width;     // f64 per body (globals: 1)
    bool global;        // tick / simulation_time_step: one 8-byte scalar, host resident
    double *dev;        // width planes of ld doubles
};

inline uint64_t round_up(uint64_t x, uint64_t m) { return (x + m - 1) / m * m; }

// A per-tick input table bound to one effector input column (b200_sixdof_set_schedule).  Row r, plane p lives at
// table + (r*width + p)*ld: every row is laid out like the column itself.
struct Schedule {
    uint64_t id;
    uint32_t width;
    double *table;
    uint64_t n_rows, first_tick;
    bool pending = false; // ticks ran since the column last received a row: it still holds an older value
    uint64_t last_tick = 0; // Tick value of the last integrated tick (the row the column reads back as)
};

} // namespace b200

struct b200_sixdof {
    uint64_t serial = 0;               // unique per created handle: what a peer window remembers of its owner besides the address
    b200_sixdof_desc desc{};
    std::vector<b200_effector> effectors;
    std::vector<uint8_t *> eff_masks; // device copies of the per-effector entity masks (nullptr = all)
    std::vector<double *> eff_tables; // device tables of GRAVITY_EGM08 effectors (nullptr = none)
    int egm_eff = -1;                  // index of the GRAVITY_EGM08 effector (at most one), -1 = none
    double *aforce = nullptr;          // 9 planes of additive stage forces it fills every tick
    int device = 0;
    uint64_t n_bodies = 0;
    uint64_t ld = 0;
    std::vector<b200::Column> cols;
    std::vector<b200::Schedule> schedules; // input schedules, at most one per effector input column
    std::vector<uint64_t> input_ids, output_ids;
    double sim_time_step = 0.0;   // SimulationTimeStep column value
    uint64_t tick = 0;            // Tick column value
    uint64_t ticks_done = 0;      // ticks since create / trajectory reset (trajectory slot index base)
    // graph effector
    int graph_eff = -1;
    bool graph_dense = false;
    uint32_t *row_ptr = nullptr, *col_idx = nullptr;
    uint8_t *has_edge = nullptr;
    double *gforce = nullptr;
    double *pos_alt = nullptr, *vel_alt = nullptr; // ping-pong planes of the one-launch n-body tick
    bool nbody_fused = false;                       // decided once per handle (whole-batch grid size)
    bool small_world = false;                       // <= 32 bodies per world: whole ticks in one warp, n ticks per launch
    uint32_t max_deg = 0;
    // staging for AoS <-> SoA
    double *staging = nullptr;
    uint64_t staging_bytes = 0;
    // trajectory
    double *traj = nullptr;
    uint32_t traj_planes = 13;   // 25 with B200_TRAJ_FULL
    // plumbing
    cudaStream_t stream = nullptr;
    bool own_stream = true;
    // pipelined invoke_batch: copy engines on their own streams, whole-batch AoS staging
    cudaStream_t copy_in = nullptr, copy_out = nullptr;
    double *stage_in = nullptr, *stage_out = nullptr;
    uint64_t stage_in_bytes = 0, stage_out_bytes = 0;
    std::vector<cudaEvent_t> chunk_in, chunk_out;
    // small batches: packed pinned host staging (one PCIe transfer per direction)
    uint8_t *host_pack = nullptr;
    uint64_t host_pack_bytes = 0;
    cudaEvent_t ev[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr}; // [0,1] H2D span, [2,3] compute span, [4,5] D2H span
    int status = B200_OK;
    b200_timings timings{};

    b200::Column *find(uint64_t id)
    {
        for (auto &c : cols) if (c.id == id) return &c;
        return nullptr;
    }
    const b200::Column *find(uint64_t id) const
    {
        for (auto &c : cols) if (c.id == id) return &c;
        return nullptr;
    }
    b200::Schedule *find_schedule(uint64_t id)
    {
        for (auto &s : schedules) if (s.id == id) return &s;
        return nullptr;
    }
};


namespace b200 {

int cuda_fail(b200_sixdof *h, cudaError_t e, const char *what);
int ensure_staging(b200_sixdof *h, uint64_t bytes);
void fill_step_params(b200_sixdof *h, StepParams &P); // every plane base, constant and effector of the handle

#define CU(h, call)                                                        \
    do {                                                                   \
        cudaError_t e_ = (call);                                           \
        if (e_ != cudaSuccess) return b200::cuda_fail((h), e_, #call);     \
    } while (0)

} // namespace b200
