// Host runtime + C ABI of libb200_sixdof (include/b200_sixdof.h).
//
// Replaces CraneliftExec (libs/nox-py/src/cranelift_exec.rs:54-195) on the
// six_dof() path: owns device-resident SoA columns, maps the reference's host
// column buffers in and out, and drives the sm_100a kernels.  There is no CPU
// fallback anywhere in this file: without a CUDA device every entry point fails
// with B200_ERR_NO_DEVICE.
#include <sys/mman.h>
#include <sys/syscall.h>
#include <unistd.h>

#include <algorithm>
#include <atomic>
#include <cctype>
#include <chrono>
#include <map>
#include <mutex>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include <thread>
#include <vector>

#include "sixdof_handle.h"

using namespace b200;

namespace b200 {

static thread_local std::string g_last_error = "";

int fail(int code, const char *fmt, ...)
{
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_last_error = buf;
    return code;
}

const char *last_error_message() { return g_last_error.c_str(); }

int cuda_fail(b200_sixdof *h, cudaError_t e, const char *what)
{
    if (h) h->status = B200_ERR_CUDA;
    return fail(e == cudaErrorMemoryAllocation ? B200_ERR_OUT_OF_MEMORY : B200_ERR_CUDA, "CUDA error in %s: %s", what,
                cudaGetErrorString(e));
}

int ensure_staging(b200_sixdof *h, uint64_t bytes)
{
    if (h->staging_bytes >= bytes) return B200_OK;
    if (h->staging) { CU(h, cudaFree(h->staging)); h->staging = nullptr; h->staging_bytes = 0; }
    CU(h, cudaMalloc(&h->staging, bytes));
    h->staging_bytes = bytes;
    return B200_OK;
}

} // namespace b200

namespace {

thread_local b200_sixdof *g_tick_handle = nullptr;

uint64_t column_bytes(const b200_sixdof *h, const Column &c)
{
    return c.global ? 8ull : h->n_bodies * c.width * 8ull;
}

// The reference's free six_dof() system has inputs (first-init order)
//   tick, force, inertia, world_pos, world_accel, simulation_time_step, world_vel
// (SURVEY §8a-7, cranelift-mlir/tests/three_body_e2e.rs:15-16); effector
// columns are inserted after `force` in effector order.  Outputs are every
// variable of the builder, ordered by ComponentId (BTreeMap, system.rs).
void build_id_tables(b200_sixdof *h)
{
    std::vector<uint64_t> in = {B200_ID_TICK, B200_ID_FORCE};
    for (auto &e : h->effectors)
        if (e.column_id && std::find(in.begin(), in.end(), e.column_id) == in.end()) in.push_back(e.column_id);
    for (uint64_t id : {B200_ID_INERTIA, B200_ID_WORLD_POS, B200_ID_WORLD_ACCEL, B200_ID_SIMULATION_TIME_STEP,
                        B200_ID_WORLD_VEL})
        if (std::find(in.begin(), in.end(), id) == in.end()) in.push_back(id);
    h->input_ids = in;
    h->output_ids = in;
    std::sort(h->output_ids.begin(), h->output_ids.end());
}

int add_column(b200_sixdof *h, uint64_t id, uint32_t width, bool global)
{
    if (h->find(id)) return B200_OK;
    Column c{id, width, global, nullptr};
    if (!global && h->n_bodies) {
        const uint64_t bytes = (uint64_t)width * h->ld * 8ull;
        CU(h, cudaMalloc(&c.dev, bytes));
        CU(h, cudaMemsetAsync(c.dev, 0, bytes, h->stream));
    }
    h->cols.push_back(c);
    return B200_OK;
}

// Derived tables of the EGM08 recursion (python/elodin/egm08.py:84-144) — the same formulas, operation for operation,
// as the test oracle's orc_egm08_tables, so both sides evaluate the series on bit-identical constants — emitted as ONE
// stream in the order egm08_field consumes it: column by column (m = 0..L), degree by degree (l = m..L), eight doubles
// per term:
//   [0] the A recursion's first constant: diag[m] (l = m), offc[l] (l = m+1), n1[l][m] otherwise      [1] n2[l][m] or 0
//   [2] the same for B at (l+1, m+1): diag[m+1], offc[l+1], n1[l+1][m+1], or 0 beyond degree L         [3] n2[l+1][m+1] or 0
//   [4] C[l][m]   [5] S[l][m]   [6] nq1[l][m]   [7] nq2[l][m]
// so a warp reads the 137 KB of a degree-64 field front to back, 64 contiguous bytes per term.
double kdelta(int d) { return d == 0 ? 1.0 : 2.0; }

std::vector<double> egm08_tables(int L, const double *c_bar, const double *s_bar)
{
    const int n = L + 1;
    std::vector<double> n1((size_t)n * n, 0.0), n2((size_t)n * n, 0.0), nq1((size_t)n * n, 0.0), nq2((size_t)n * n, 0.0), diag(n), offc(n);
    for (int l = 0; l <= L; ++l)
        for (int m = 0; m <= L; ++m) {
            double v1 = 0.0, v2 = 0.0;
            if (l >= m + 2) {
                v1 = std::sqrt((double)((2 * l + 1) * (2 * l - 1)) / (double)((l + m) * (l - m)));
                v2 = std::sqrt((double)((l + m - 1) * (l - m - 1) * (2 * l + 1)) / (double)((2 * l - 3) * (l + m) * (l - m)));
            }
            n1[l * n + m] = v1;
            n2[l * n + m] = v2;
            const double num1 = (double)(l - m) * kdelta(m) * (double)(l + m + 1);
            nq1[l * n + m] = num1 < 0.0 ? 0.0 : std::sqrt(num1 / kdelta(m + 1));
            const double num2 = (double)(l + m + 2) * (double)(l + m + 1) * (double)(2 * l + 1) * kdelta(m);
            nq2[l * n + m] = num2 < 0.0 ? 0.0 : std::sqrt(num2 / ((double)(2 * l + 3) * kdelta(m + 1)));
        }
    double cur = 1.0;
    for (int l = 0; l <= L; ++l) {
        if (l > 0) cur = cur * std::sqrt(((double)(2 * l + 1) * kdelta(l)) / ((double)(2 * l) * kdelta(l - 1)));
        diag[l] = cur;
        offc[l] = l == 0 ? 0.0 : diag[l] * std::sqrt(((double)(2 * l) * kdelta(l - 1)) / kdelta(l));
    }
    std::vector<double> t;
    t.reserve((size_t)4 * n * (n + 1));
    for (int m = 0; m <= L; ++m)
        for (int l = m; l <= L; ++l) {
            const int l1 = l + 1, m1 = m + 1;
            const bool b_live = m1 <= L && l1 <= L;
            t.push_back(l == m ? diag[m] : l == m + 1 ? offc[l] : n1[l * n + m]);
            t.push_back(l >= m + 2 ? n2[l * n + m] : 0.0);
            t.push_back(!b_live ? 0.0 : l1 == m1 ? diag[m1] : l1 == m1 + 1 ? offc[l1] : n1[l1 * n + m1]);
            t.push_back(b_live && l1 >= m1 + 2 ? n2[l1 * n + m1] : 0.0);
            t.push_back(c_bar[l * n + m]);
            t.push_back(s_bar[l * n + m]);
            t.push_back(nq1[l * n + m]);
            t.push_back(nq2[l * n + m]);
        }
    return t;
}

int build_graph(b200_sixdof *h, const b200_effector &e)
{
    const uint32_t N = (uint32_t)h->desc.n_entities;
    std::vector<uint32_t> row(N + 1, 0), col;
    std::vector<std::vector<uint32_t>> adj(N);
    for (uint64_t k = 0; k < e.n_edges; ++k) {
        const uint32_t a = e.edge_from[k], b = e.edge_to[k];
        if (a >= N || b >= N) return fail(B200_ERR_INVALID_ARGUMENT, "edge %llu (%u -> %u) out of range (n_entities=%u)",
                                          (unsigned long long)k, a, b, N);
        adj[a].push_back(b); // spawn order preserved per source (graph.rs:194-197)
    }
    std::vector<uint8_t> has(N ? N : 1, 0);
    bool dense = N > 1;
    for (uint32_t i = 0; i < N; ++i) {
        row[i + 1] = row[i] + (uint32_t)adj[i].size();
        col.insert(col.end(), adj[i].begin(), adj[i].end());
        has[i] = !adj[i].empty();
        if (adj[i].size() != N - 1) dense = false;
        else {
            uint32_t want = 0;
            for (uint32_t t : adj[i]) { if (want == i) ++want; if (t != want) { dense = false; break; } ++want; }
        }
    }
    h->graph_dense = dense;
    for (uint32_t i = 0; i < N; ++i) h->max_deg = std::max<uint32_t>(h->max_deg, (uint32_t)adj[i].size());
    CU(h, cudaMalloc(&h->row_ptr, (N + 1) * sizeof(uint32_t)));
    CU(h, cudaMalloc(&h->col_idx, std::max<size_t>(col.size(), 1) * sizeof(uint32_t)));
    CU(h, cudaMalloc(&h->has_edge, has.size()));
    CU(h, cudaMemcpy(h->row_ptr, row.data(), (N + 1) * sizeof(uint32_t), cudaMemcpyHostToDevice));
    if (!col.empty()) CU(h, cudaMemcpy(h->col_idx, col.data(), col.size() * sizeof(uint32_t), cudaMemcpyHostToDevice));
    CU(h, cudaMemcpy(h->has_edge, has.data(), has.size(), cudaMemcpyHostToDevice));
    CU(h, cudaMalloc(&h->gforce, 9ull * h->ld * 8ull));
    CU(h, cudaMemset(h->gforce, 0, 9ull * h->ld * 8ull));
    if (h->desc.math_mode == B200_MATH_FAST && dense) {
        CU(h, cudaMalloc(&h->pos_alt, 7ull * h->ld * 8ull));
        CU(h, cudaMalloc(&h->vel_alt, 6ull * h->ld * 8ull));
        CU(h, cudaMemset(h->pos_alt, 0, 7ull * h->ld * 8ull));
        CU(h, cudaMemset(h->vel_alt, 0, 6ull * h->ld * 8ull));
    }
    return B200_OK;
}

} // namespace

namespace b200 {

void fill_step_params(b200_sixdof *h, StepParams &P)
{
    std::memset(&P, 0, sizeof P);
    P.pos = h->find(B200_ID_WORLD_POS)->dev;
    P.vel = h->find(B200_ID_WORLD_VEL)->dev;
    P.acc = h->find(B200_ID_WORLD_ACCEL)->dev;
    P.frc = h->find(B200_ID_FORCE)->dev;
    P.ine = h->find(B200_ID_INERTIA)->dev;
    P.gforce = h->gforce;
    P.has_edge = h->has_edge;
    P.aforce = h->aforce;
    P.ld = h->ld;
    P.n_bodies = h->n_bodies;
    P.n_entities = (uint32_t)h->desc.n_entities;
    P.n_eff = (uint32_t)h->effectors.size();
    P.dt_stage = h->sim_time_step;
    P.dt_final = std::isnan(h->desc.time_step) ? h->sim_time_step : h->desc.time_step;
    P.traj = h->traj;
    P.traj_capacity = h->desc.trajectory_capacity;
    P.traj_every = h->traj ? h->desc.trajectory_every : 0;
    P.traj_planes = h->traj_planes;
    for (size_t i = 0; i < h->effectors.size(); ++i) {
        const b200_effector &e = h->effectors[i];
        P.eff[i].kind = e.kind;
        P.eff[i].flags = e.flags;
        std::memcpy(P.eff[i].p, e.p, sizeof e.p);
        const Column *c = e.column_id ? h->find(e.column_id) : nullptr;
        P.eff[i].col = c ? c->dev : nullptr;
        P.eff[i].col_width = c ? c->width : 0;
        P.eff[i].mask = i < h->eff_masks.size() ? h->eff_masks[i] : nullptr;
        P.eff[i].table = i < h->eff_tables.size() ? h->eff_tables[i] : nullptr;
    }
}

} // namespace b200

namespace {

bool is_state_column(uint64_t id)
{
    return id == B200_ID_WORLD_POS || id == B200_ID_WORLD_VEL || id == B200_ID_WORLD_ACCEL || id == B200_ID_FORCE ||
           id == B200_ID_INERTIA || id == B200_ID_TICK || id == B200_ID_SIMULATION_TIME_STEP;
}

// Point every scheduled effector column of a launch of n ticks, the first of which has Tick value `tick`, at its
// table.  One tick reads one fixed row: the kernels see a plain column and every existing instantiation applies.
// Several ticks carry the row stride and the row rule; the kernels compiled for it read each tick's own row.
void bind_schedules(b200_sixdof *h, StepParams &P, uint64_t b0, uint64_t n, uint64_t tick)
{
    P.tick_abs = tick;
    P.sched = 0;
    if (h->schedules.empty()) return;
    for (uint32_t i = 0; i < P.n_eff; ++i) {
        const uint64_t id = h->effectors[i].column_id;
        const Schedule *s = id ? h->find_schedule(id) : nullptr;
        if (!s) continue;
        const uint64_t stride = (uint64_t)s->width * h->ld;
        if (n == 1) {
            P.eff[i].col = s->table + schedule_row(tick, s->first_tick, s->n_rows) * stride + b0;
            P.eff[i].sched = SchedDev{0, 0, 0};
        } else {
            P.eff[i].col = s->table + b0;
            P.eff[i].sched = SchedDev{stride, s->n_rows, s->first_tick};
            P.sched = 1;
        }
    }
}

// After n ticks the scheduled columns read back as the row of the last one; the copy waits until someone reads them
void note_schedule_ticks(b200_sixdof *h, uint64_t n_ticks)
{
    if (n_ticks == 0) return;
    for (auto &s : h->schedules) { s.pending = true; s.last_tick = h->tick - 1; }
}

int materialise_schedule(b200_sixdof *h, Schedule &s)
{
    if (!s.pending) return B200_OK;
    const uint64_t stride = (uint64_t)s.width * h->ld;
    if (h->n_bodies)
        CU(h, cudaMemcpyAsync(h->find(s.id)->dev, s.table + schedule_row(s.last_tick, s.first_tick, s.n_rows) * stride,
                              stride * 8ull, cudaMemcpyDeviceToDevice, h->stream));
    s.pending = false;
    return B200_OK;
}

// Integrate n_ticks ticks of the worlds [w0, w0+nw) on `stream`.  Worlds are independent, so a
// world range can run to completion before the next one starts (used by the pipelined
// invoke_batch); counters are the caller's business.
int launch_ticks(b200_sixdof *h, uint64_t w0, uint64_t nw, uint64_t n_ticks, cudaStream_t stream)
{
    const uint64_t N = h->desc.n_entities;
    const uint64_t b0 = w0 * N, nb = nw * N;
    if (n_ticks == 0 || nb == 0) return B200_OK;
    StepParams P;
    fill_step_params(h, P);
    // shift every per-body plane base to the range start; rows inside a world keep their index
    P.pos += b0; P.vel += b0; P.acc += b0; P.frc += b0; P.ine += b0;
    if (P.gforce) P.gforce += b0;
    if (P.aforce) P.aforce += b0;
    if (P.traj) P.traj += b0;
    for (uint32_t i = 0; i < P.n_eff; ++i) if (P.eff[i].col) P.eff[i].col += b0;
    P.n_bodies = nb;
    const bool exact = h->desc.math_mode == B200_MATH_EXACT;
    const bool graph = h->graph_eff >= 0;
    const bool egm = h->egm_eff >= 0; // its stage forces are a function of the tick's input state: one launch per tick
    const uint64_t fuse = ((graph && !h->small_world) || egm) ? 1 : std::max<uint32_t>(1u, h->desc.max_fused_ticks);
    uint64_t left = n_ticks, done = 0;
    double *pos_next = h->pos_alt ? h->pos_alt + b0 : nullptr, *vel_next = h->vel_alt ? h->vel_alt + b0 : nullptr;
    while (left) {
        const uint64_t n = std::min(left, fuse);
        bind_schedules(h, P, b0, n, h->tick + done);
        if (egm) {
            const b200_effector &ge = h->effectors[h->egm_eff];
            EgmParams E{};
            E.pos = P.pos; E.vel = P.vel; E.ine = P.ine; E.aforce = h->aforce + b0;
            E.table = h->eff_tables[h->egm_eff]; E.mask = h->eff_masks[h->egm_eff];
            E.ld = h->ld; E.n_bodies = nb; E.n_entities = P.n_entities; E.ent0 = 0;
            E.L = (uint32_t)ge.p[2]; E.integrator = h->desc.integrator; E.mu = ge.p[0]; E.r_ref = ge.p[1]; E.dt_stage = P.dt_stage;
            CU(h, launch_egm08_force(E, (int)h->desc.math_mode, stream));
            h->timings.kernel_launches++;
        }
        if (graph) {
            const b200_effector &e = h->effectors[h->graph_eff];
            GraphParams G{};
            G.pos = P.pos; G.vel = P.vel; G.ine = P.ine; G.gforce = h->gforce + b0;
            G.ld = h->ld; G.n_entities = P.n_entities; G.n_worlds = (uint32_t)nw;
            G.dt_stage = P.dt_stage; G.kind = e.kind; G.integrator = h->desc.integrator;
            G.p0 = e.p[0]; G.p1 = e.p[1]; G.row_ptr = h->row_ptr; G.col_idx = h->col_idx; G.max_deg = h->max_deg;
            if (h->small_world) {
                // gravity through warp shuffles + integration, n ticks in one launch, state in registers
                P.n_ticks = (uint32_t)n;
                P.tick0 = h->ticks_done + done;
                P.write_fa = (exact || left == n) ? 1u : 0u;
                CU(h, launch_small_world(G, P, (int)h->desc.math_mode, stream));
                h->timings.kernel_launches++;
                done += n;
                left -= n;
                continue;
            }
            if (h->nbody_fused) {
                // gravity + integration in one launch; the new state lands in the other plane set
                P.n_ticks = 1;
                P.tick0 = h->ticks_done + done;
                P.write_fa = (left == 1) ? 1u : 0u;
                CU(h, launch_nbody_tick_fused(G, P, pos_next, vel_next, stream));
                h->timings.kernel_launches++;
                std::swap(P.pos, pos_next);
                std::swap(P.vel, vel_next);
                done += 1;
                left -= 1;
                continue;
            }
            CU(h, launch_graph_force(G, h->desc.math_mode, h->graph_dense, stream));
            h->timings.kernel_launches++;
        }
        P.n_ticks = (uint32_t)n;
        P.tick0 = h->ticks_done + done;
        P.write_fa = (exact || left == n) ? 1u : 0u; // Force/WorldAccel are only host-visible after the batch
        P.reverse = (uint32_t)(h->timings.kernel_launches & 1u); // alternate the traversal direction launch to launch
        CU(h, launch_body_step(P, (int)h->desc.integrator, (int)h->desc.math_mode, stream));
        h->timings.kernel_launches++;
        done += n;
        left -= n;
    }
    return B200_OK;
}

// After every world range has advanced n_ticks through the one-launch n-body tick, the live pose /
// velocity planes are the "other" set when n_ticks is odd: make them the columns' planes.
void commit_ping_pong(b200_sixdof *h, uint64_t n_ticks)
{
    if (!h->nbody_fused || !(n_ticks & 1) || h->n_bodies == 0) return;
    std::swap(h->find(B200_ID_WORLD_POS)->dev, h->pos_alt);
    std::swap(h->find(B200_ID_WORLD_VEL)->dev, h->vel_alt);
}

int do_step(b200_sixdof *h, uint64_t n_ticks)
{
    if (h->status != B200_OK) return fail(h->status, "handle is in a failed state");
    int rc = launch_ticks(h, 0, h->desc.n_worlds, n_ticks, h->stream);
    if (rc) return rc;
    commit_ping_pong(h, n_ticks);
    h->ticks_done += n_ticks;
    h->tick += n_ticks;
    h->timings.ticks += n_ticks;
    note_schedule_ticks(h, n_ticks);
    return B200_OK;
}

int do_upload(b200_sixdof *h, uint64_t id, const void *src, uint64_t bytes)
{
    Column *c = h->find(id);
    if (!c) return fail(B200_ERR_COMPONENT_NOT_FOUND, "component not found: 0x%016llx", (unsigned long long)id);
    if (bytes != column_bytes(h, *c))
        return fail(B200_ERR_VALUE_SIZE_MISMATCH, "component value had wrong size: 0x%016llx has %llu bytes, got %llu",
                    (unsigned long long)id, (unsigned long long)column_bytes(h, *c), (unsigned long long)bytes);
    if (!src) return fail(B200_ERR_INVALID_ARGUMENT, "null source buffer");
    if (h->find_schedule(id))
        return fail(B200_ERR_INVALID_ARGUMENT, "column 0x%016llx is driven by an input schedule (clear it to upload)",
                    (unsigned long long)id);
    if (c->global) {
        // the two globals are 8-byte host scalars (Globals entity, world.rs:174-191)
        uint64_t raw;
        std::memcpy(&raw, src, 8);
        if (id == B200_ID_TICK) h->tick = raw;
        else std::memcpy(&h->sim_time_step, &raw, 8);
        return B200_OK;
    }
    if (bytes == 0) return B200_OK;
    int rc = ensure_staging(h, bytes);
    if (rc) return rc;
    CU(h, cudaMemcpyAsync(h->staging, src, bytes, cudaMemcpyDefault, h->stream));
    CU(h, launch_aos_to_soa(h->staging, c->dev, h->n_bodies, c->width, h->ld, h->stream));
    h->timings.kernel_launches++;
    return B200_OK;
}

int do_download(b200_sixdof *h, uint64_t id, void *dst, uint64_t bytes)
{
    Column *c = h->find(id);
    if (!c) return fail(B200_ERR_COMPONENT_NOT_FOUND, "component not found: 0x%016llx", (unsigned long long)id);
    if (bytes != column_bytes(h, *c))
        return fail(B200_ERR_VALUE_SIZE_MISMATCH, "component value had wrong size: 0x%016llx has %llu bytes, got %llu",
                    (unsigned long long)id, (unsigned long long)column_bytes(h, *c), (unsigned long long)bytes);
    if (!dst) return fail(B200_ERR_INVALID_ARGUMENT, "null destination buffer");
    if (c->global) {
        uint64_t raw;
        if (id == B200_ID_TICK) raw = h->tick;
        else std::memcpy(&raw, &h->sim_time_step, 8);
        std::memcpy(dst, &raw, 8);
        return B200_OK;
    }
    if (bytes == 0) return B200_OK;
    int rc = B200_OK;
    if (Schedule *s = h->find_schedule(id)) if ((rc = materialise_schedule(h, *s))) return rc;
    if ((rc = ensure_staging(h, bytes))) return rc;
    CU(h, launch_soa_to_aos(c->dev, h->staging, h->n_bodies, c->width, h->ld, h->stream));
    h->timings.kernel_launches++;
    CU(h, cudaMemcpyAsync(dst, h->staging, bytes, cudaMemcpyDefault, h->stream));
    // the staging buffer is reused by the next transfer; the copy must have left it first
    CU(h, cudaStreamSynchronize(h->stream));
    return B200_OK;
}

float ev_ms(cudaEvent_t a, cudaEvent_t b)
{
    float ms = 0.f;
    cudaEventElapsedTime(&ms, a, b);
    return ms;
}

} // namespace

// ===================================================================== C ABI

extern "C" {

uint64_t b200_component_id(const char *name)
{
    uint64_t h = 0xcbf29ce484222325ull; // FNV-1a 64 offset basis
    if (name)
        for (const unsigned char *p = (const unsigned char *)name; *p; ++p) { h ^= *p; h *= 0x100000001b3ull; }
    return h & ~(1ull << 63); // types.rs:43
}

const char *b200_last_error(void) { return last_error_message(); }

int b200_device_count(void)
{
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) { (void)cudaGetLastError(); return -fail(B200_ERR_NO_DEVICE, "no CUDA device: %s", cudaGetErrorString(e)); }
    return n;
}

void *b200_host_alloc(uint64_t bytes)
{
    void *p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocDefault) != cudaSuccess) {
        fail(B200_ERR_OUT_OF_MEMORY, "cudaHostAlloc(%llu) failed: %s", (unsigned long long)bytes,
             cudaGetErrorString(cudaGetLastError()));
        return nullptr;
    }
    return p;
}

// NUMA node of a GPU's PCIe root: /sys/bus/pci/devices/<domain:bus:dev.fn>/numa_node
int b200_device_numa_node(int device)
{
    char bus[32] = {0};
    if (cudaDeviceGetPCIBusId(bus, sizeof bus, device) != cudaSuccess) { (void)cudaGetLastError(); return -1; }
    for (char *c = bus; *c; ++c) *c = (char)std::tolower((unsigned char)*c);
    char path[128];
    snprintf(path, sizeof path, "/sys/bus/pci/devices/%s/numa_node", bus);
    FILE *f = fopen(path, "r");
    if (!f) return -1;
    int node = -1;
    if (fscanf(f, "%d", &node) != 1) node = -1;
    fclose(f);
    return node;
}

// NUMA node the first page of a host buffer lives on (move_pages query), -1 if unknown
int b200_host_node_of(const void *p)
{
#ifdef SYS_move_pages
    void *page = (void *)((uintptr_t)p & ~(uintptr_t)4095);
    int status = -1;
    if (syscall(SYS_move_pages, 0, 1ul, &page, nullptr, &status, 0) == 0) return status;
#endif
    return -1;
}

namespace {
std::mutex g_local_mu;
std::map<void *, size_t> g_local_allocs; // b200_host_alloc_local blocks: base -> mapped length
}

// Page-locked host memory on the NUMA node of `device`'s PCIe root: anonymous mapping, mbind(MPOL_BIND) to that
// node, first touch, cudaHostRegister.  With 4 GPUs per socket moving ~100 GB/s each way, buffers that sit on the
// other socket (or interleaved) make the inter-socket link the bottleneck.  Falls back to b200_host_alloc when the
// node is unknown or the policy cannot be applied.
void *b200_host_alloc_local(uint64_t bytes, int device)
{
    if (device < 0 && cudaGetDevice(&device) != cudaSuccess) { (void)cudaGetLastError(); return b200_host_alloc(bytes); }
    const int node = b200_device_numa_node(device);
    if (node < 0 || node >= 1024) return b200_host_alloc(bytes);
    const size_t len = (size_t)round_up(std::max<uint64_t>(bytes, 1), 2ull << 20);
    void *p = mmap(nullptr, len, PROT_READ | PROT_WRITE, MAP_PRIVATE | MAP_ANONYMOUS, -1, 0);
    if (p == MAP_FAILED) return b200_host_alloc(bytes);
#ifdef SYS_mbind
    unsigned long mask[16] = {0};
    mask[node / (8 * sizeof(unsigned long))] |= 1ul << (node % (8 * sizeof(unsigned long)));
    if (syscall(SYS_mbind, p, len, 2 /* MPOL_BIND */, mask, sizeof mask * 8, 0u) != 0) {
        munmap(p, len); // the node is not in this process's allowed set: plain first-touch allocation instead
        return b200_host_alloc(bytes);
    }
#endif
    std::memset(p, 0, len); // first touch under the policy
    if (cudaHostRegister(p, len, cudaHostRegisterDefault) != cudaSuccess) {
        (void)cudaGetLastError();
        munmap(p, len);
        return b200_host_alloc(bytes);
    }
    std::lock_guard<std::mutex> lock(g_local_mu);
    g_local_allocs[p] = len;
    return p;
}

void b200_host_free(void *p)
{
    if (!p) return;
    {
        std::lock_guard<std::mutex> lock(g_local_mu);
        auto it = g_local_allocs.find(p);
        if (it != g_local_allocs.end()) {
            cudaHostUnregister(p);
            munmap(p, it->second);
            g_local_allocs.erase(it);
            return;
        }
    }
    cudaFreeHost(p);
}

int b200_sixdof_create(const b200_sixdof_desc *d, b200_sixdof **out)
{
    if (!d || !out) return fail(B200_ERR_INVALID_ARGUMENT, "null descriptor / out pointer");
    *out = nullptr;
    if (d->abi_version != B200_SIXDOF_ABI_VERSION)
        return fail(B200_ERR_INVALID_ARGUMENT, "ABI version mismatch: library %u, caller %u", B200_SIXDOF_ABI_VERSION,
                    d->abi_version);
    if (d->integrator > B200_INTEGRATOR_SEMI_IMPLICIT) return fail(B200_ERR_UNSUPPORTED, "unknown integrator %u", d->integrator);
    if (d->math_mode > B200_MATH_FAST) return fail(B200_ERR_UNSUPPORTED, "unknown math mode %u", d->math_mode);
    if (d->n_effectors > B200_MAX_EFFECTORS) return fail(B200_ERR_UNSUPPORTED, "too many effectors (%u > %u)", d->n_effectors, B200_MAX_EFFECTORS);
    if (d->n_effectors && !d->effectors) return fail(B200_ERR_INVALID_ARGUMENT, "n_effectors > 0 but effectors is null");
    if (d->n_worlds == 0) return fail(B200_ERR_INVALID_ARGUMENT, "n_worlds must be >= 1");
    if (d->n_entities > 0xffffffffull || d->n_worlds > 0xffffffffull) return fail(B200_ERR_UNSUPPORTED, "n_entities / n_worlds exceed 2^32-1");
    if ((d->trajectory_flags & ~(uint32_t)B200_TRAJ_FULL) || d->reserved0)
        return fail(B200_ERR_INVALID_ARGUMENT, "unknown trajectory_flags 0x%x / non-zero reserved field", d->trajectory_flags);
    if (!(d->sim_time_step > 0.0) || !std::isfinite(d->sim_time_step))
        return fail(B200_ERR_INVALID_ARGUMENT, "invalid time step: %g", d->sim_time_step); // Error::InvalidTimeStep

    int ndev = b200_device_count();
    if (ndev <= 0) return fail(B200_ERR_NO_DEVICE, "no CUDA device visible; this library has no CPU fallback");
    int dev = d->device;
    if (dev < 0) { if (cudaGetDevice(&dev) != cudaSuccess) dev = 0; }
    if (dev >= ndev) return fail(B200_ERR_INVALID_ARGUMENT, "device %d out of range (%d devices)", dev, ndev);

    b200_sixdof *h = new (std::nothrow) b200_sixdof();
    if (!h) return fail(B200_ERR_OUT_OF_MEMORY, "out of host memory");
    static std::atomic<uint64_t> next_serial{1};
    h->serial = next_serial.fetch_add(1);
    h->desc = *d;
    h->device = dev;
    h->effectors.assign(d->effectors, d->effectors + d->n_effectors);
    h->desc.effectors = nullptr;
    h->n_bodies = d->n_entities * d->n_worlds;
    h->ld = round_up(std::max<uint64_t>(h->n_bodies, 1), 128); // whole 128-body tiles inside every plane
    h->sim_time_step = d->sim_time_step;

    int rc = B200_OK;
    auto bail = [&](int code) { b200_sixdof_destroy(h); return code; };
    if (cudaSetDevice(dev) != cudaSuccess) return bail(cuda_fail(nullptr, cudaGetLastError(), "cudaSetDevice"));
    if (cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking) != cudaSuccess)
        return bail(cuda_fail(nullptr, cudaGetLastError(), "cudaStreamCreate"));
    for (auto &e : h->ev)
        if (cudaEventCreate(&e) != cudaSuccess) return bail(cuda_fail(nullptr, cudaGetLastError(), "cudaEventCreate"));

    // validate effectors
    int n_drag = 0, n_frame = 0;
    for (size_t i = 0; i < h->effectors.size(); ++i) {
        b200_effector &e = h->effectors[i];
        uint32_t want_w = 0;
        switch (e.kind) {
        case B200_EFF_GRAVITY_CONST: case B200_EFF_GRAVITY_FRAME: want_w = 0; break;
        case B200_EFF_DRAG_QUADRATIC: want_w = 3; ++n_drag; break;
        case B200_EFF_THRUST_BODY: want_w = 1; break;
        case B200_EFF_WRENCH_BODY: case B200_EFF_WRENCH_WORLD: want_w = 6; break;
        case B200_EFF_GRAVITY_J2: want_w = 0; break;
        case B200_EFF_GRAVITY_EGM08: {
            want_w = 0;
            const double Ld = e.p[2];
            if (!(Ld >= 0.0) || Ld > 128.0 || Ld != std::floor(Ld))
                return bail(fail(B200_ERR_INVALID_ARGUMENT, "effector %zu: EGM08 max_degree must be an integer in 0..128 (got %g)", i, Ld));
            const uint64_t n = (uint64_t)Ld + 1;
            if (!e.table0 || !e.table1 || e.table_len != n * n)
                return bail(fail(B200_ERR_VALUE_SIZE_MISMATCH, "effector %zu: EGM08 needs C and S tables of (L+1)^2 = %llu f64 (got %llu)", i,
                                 (unsigned long long)(n * n), (unsigned long long)e.table_len));
            if (h->egm_eff >= 0) return bail(fail(B200_ERR_UNSUPPORTED, "only one EGM08 gravity effector is supported"));
            h->egm_eff = (int)i;
            break;
        }
        case B200_EFF_TORQUE_BODY_FOLD:
            want_w = e.column_width; // 3 per wheel
            if (e.column_width == 0 || e.column_width % 3 != 0 || e.column_width > 24)
                return bail(fail(B200_ERR_VALUE_SIZE_MISMATCH, "effector %zu: a wheel-torque column holds 3 f64 per wheel, 1..8 wheels (got width %u)", i, e.column_width));
            break;
        case B200_EFF_GRAVITY_EDGES_NEWTON: case B200_EFF_GRAVITY_EDGES_SOFTENED:
            if (h->graph_eff >= 0) return bail(fail(B200_ERR_UNSUPPORTED, "only one edge_fold gravity effector is supported"));
            if (e.n_edges && (!e.edge_from || !e.edge_to)) return bail(fail(B200_ERR_INVALID_ARGUMENT, "edge arrays are null"));
            if (d->math_mode == B200_MATH_FAST && i != 0)
                return bail(fail(B200_ERR_UNSUPPORTED, "FAST math: the edge_fold gravity effector must come first (it overwrites Force)"));
            h->graph_eff = (int)i;
            break;
        default:
            return bail(fail(B200_ERR_UNSUPPORTED, "effector kind %u is not built in (no CPU fallback, no JIT)", e.kind));
        }
        if (e.kind == B200_EFF_GRAVITY_FRAME) ++n_frame;
        if (e.column_id) {
            if (e.column_width != want_w && !(e.kind == B200_EFF_DRAG_QUADRATIC && e.column_width == 5))
                return bail(fail(B200_ERR_VALUE_SIZE_MISMATCH, "effector %zu: column width %u, kind %u needs %u", i, e.column_width, e.kind, want_w));
        } else if (e.kind == B200_EFF_THRUST_BODY || e.kind == B200_EFF_WRENCH_BODY || e.kind == B200_EFF_WRENCH_WORLD ||
                   e.kind == B200_EFF_TORQUE_BODY_FOLD) {
            return bail(fail(B200_ERR_INVALID_ARGUMENT, "effector %zu (kind %u) needs an input column", i, e.kind));
        }
    }
    if (d->math_mode == B200_MATH_FAST && (n_drag > 1 || n_frame > 1))
        return bail(fail(B200_ERR_UNSUPPORTED, "FAST math supports at most one drag and one frame effector"));

    // columns
    if ((rc = add_column(h, B200_ID_TICK, 1, true))) return bail(rc);
    if ((rc = add_column(h, B200_ID_SIMULATION_TIME_STEP, 1, true))) return bail(rc);
    if ((rc = add_column(h, B200_ID_WORLD_POS, 7, false))) return bail(rc);
    if ((rc = add_column(h, B200_ID_WORLD_VEL, 6, false))) return bail(rc);
    if ((rc = add_column(h, B200_ID_WORLD_ACCEL, 6, false))) return bail(rc);
    if ((rc = add_column(h, B200_ID_FORCE, 6, false))) return bail(rc);
    if ((rc = add_column(h, B200_ID_INERTIA, 7, false))) return bail(rc);
    for (auto &e : h->effectors)
        if (e.column_id) {
            const Column *c = h->find(e.column_id);
            if (c && c->width != e.column_width)
                return bail(fail(B200_ERR_VALUE_SIZE_MISMATCH, "column 0x%016llx declared with two widths", (unsigned long long)e.column_id));
            if ((rc = add_column(h, e.column_id, e.column_width, false))) return bail(rc);
        }
    build_id_tables(h);
    // per-effector entity masks: copy now, the caller's arrays are only valid for this call
    h->eff_masks.assign(h->effectors.size(), nullptr);
    for (size_t i = 0; i < h->effectors.size(); ++i) {
        b200_effector &e = h->effectors[i];
        if (e.entity_mask && d->n_entities) {
            if (cudaMalloc(&h->eff_masks[i], d->n_entities) != cudaSuccess)
                return bail(cuda_fail(nullptr, cudaGetLastError(), "cudaMalloc(entity mask)"));
            if (cudaMemcpy(h->eff_masks[i], e.entity_mask, d->n_entities, cudaMemcpyHostToDevice) != cudaSuccess)
                return bail(cuda_fail(nullptr, cudaGetLastError(), "cudaMemcpy(entity mask)"));
        }
        e.entity_mask = nullptr;
    }

    // EGM08 coefficient tables: copied (with the derived recursion tables) now, the caller's arrays are only valid for this call
    h->eff_tables.assign(h->effectors.size(), nullptr);
    for (size_t i = 0; i < h->effectors.size(); ++i) {
        b200_effector &e = h->effectors[i];
        if (e.kind == B200_EFF_GRAVITY_EGM08) {
            const std::vector<double> t = egm08_tables((int)e.p[2], e.table0, e.table1);
            if (cudaMalloc(&h->eff_tables[i], t.size() * sizeof(double)) != cudaSuccess)
                return bail(cuda_fail(nullptr, cudaGetLastError(), "cudaMalloc(EGM08 tables)"));
            if (cudaMemcpy(h->eff_tables[i], t.data(), t.size() * sizeof(double), cudaMemcpyHostToDevice) != cudaSuccess)
                return bail(cuda_fail(nullptr, cudaGetLastError(), "cudaMemcpy(EGM08 tables)"));
        }
        e.table0 = e.table1 = nullptr;
    }
    if (h->graph_eff >= 0) {
        // copy the edge arrays' content now: the caller's pointers are only valid for this call
        if ((rc = build_graph(h, h->effectors[h->graph_eff]))) return bail(rc);
        {
            GraphParams G{};
            G.n_entities = (uint32_t)d->n_entities; G.n_worlds = (uint32_t)d->n_worlds; G.integrator = d->integrator;
            // (an EGM08 effector needs its stage-force launch before every body launch: the generic two-launch route)
            h->small_world = h->egm_eff < 0 && small_world_applicable(G, (int)d->math_mode);
            h->nbody_fused = h->egm_eff < 0 && !h->small_world && h->pos_alt && nbody_fused_applicable(G, (int)d->math_mode, h->graph_dense);
        }
        h->effectors[h->graph_eff].edge_from = h->effectors[h->graph_eff].edge_to = nullptr;
    }
    if (h->egm_eff >= 0) {
        if (cudaMalloc(&h->aforce, 9ull * h->ld * 8ull) != cudaSuccess) return bail(cuda_fail(nullptr, cudaGetLastError(), "cudaMalloc(EGM08 stage forces)"));
        if (cudaMemset(h->aforce, 0, 9ull * h->ld * 8ull) != cudaSuccess) return bail(cuda_fail(nullptr, cudaGetLastError(), "cudaMemset(EGM08 stage forces)"));
    }
    if (d->trajectory_every && d->trajectory_capacity) {
        h->traj_planes = (d->trajectory_flags & B200_TRAJ_FULL) ? 25u : 13u;
        if (cudaMalloc(&h->traj, d->trajectory_capacity * (uint64_t)h->traj_planes * h->ld * 8ull) != cudaSuccess)
            return bail(cuda_fail(nullptr, cudaGetLastError(), "cudaMalloc(trajectory)"));
    }
    if (cudaStreamSynchronize(h->stream) != cudaSuccess) return bail(cuda_fail(nullptr, cudaGetLastError(), "create sync"));
    *out = h;
    return B200_OK;
}

void b200_sixdof_destroy(b200_sixdof *h)
{
    if (!h) return;
    if (g_tick_handle == h) g_tick_handle = nullptr;
    cudaSetDevice(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    for (auto &c : h->cols) if (c.dev) cudaFree(c.dev);
    for (auto m : h->eff_masks) if (m) cudaFree(m);
    for (auto &s : h->schedules) if (s.table) cudaFree(s.table);
    for (auto t : h->eff_tables) if (t) cudaFree(t);
    if (h->row_ptr) cudaFree(h->row_ptr);
    if (h->col_idx) cudaFree(h->col_idx);
    if (h->has_edge) cudaFree(h->has_edge);
    if (h->gforce) cudaFree(h->gforce);
    if (h->aforce) cudaFree(h->aforce);
    if (h->pos_alt) cudaFree(h->pos_alt);
    if (h->vel_alt) cudaFree(h->vel_alt);
    if (h->staging) cudaFree(h->staging);
    if (h->stage_in) cudaFree(h->stage_in);
    if (h->stage_out) cudaFree(h->stage_out);
    if (h->traj) cudaFree(h->traj);
    for (auto &e : h->chunk_in) if (e) cudaEventDestroy(e);
    for (auto &e : h->chunk_out) if (e) cudaEventDestroy(e);
    if (h->host_pack) cudaFreeHost(h->host_pack);
    if (h->copy_in) cudaStreamDestroy(h->copy_in);
    if (h->copy_out) cudaStreamDestroy(h->copy_out);
    for (auto &e : h->ev) if (e) cudaEventDestroy(e);
    if (h->stream && h->own_stream) cudaStreamDestroy(h->stream);
    (void)cudaGetLastError();
    delete h;
}

uint32_t b200_sixdof_input_ids(const b200_sixdof *h, uint64_t *ids, uint32_t cap)
{
    if (!h) return 0;
    for (uint32_t i = 0; i < cap && i < h->input_ids.size(); ++i) ids[i] = h->input_ids[i];
    return (uint32_t)h->input_ids.size();
}

uint32_t b200_sixdof_output_ids(const b200_sixdof *h, uint64_t *ids, uint32_t cap)
{
    if (!h) return 0;
    for (uint32_t i = 0; i < cap && i < h->output_ids.size(); ++i) ids[i] = h->output_ids[i];
    return (uint32_t)h->output_ids.size();
}

uint64_t b200_sixdof_column_bytes(const b200_sixdof *h, uint64_t id)
{
    if (!h) return 0;
    const Column *c = h->find(id);
    return c ? column_bytes(h, *c) : 0;
}

int b200_sixdof_upload(b200_sixdof *h, uint64_t id, const void *src, uint64_t bytes)
{
    if (!h) return fail(B200_ERR_INVALID_ARGUMENT, "null handle");
    CU(h, cudaSetDevice(h->device));
    return do_upload(h, id, src, bytes);
}

int b200_sixdof_download(b200_sixdof *h, uint64_t id, void *dst, uint64_t bytes)
{
    if (!h) return fail(B200_ERR_INVALID_ARGUMENT, "null handle");
    CU(h, cudaSetDevice(h->device));
    return do_download(h, id, dst, bytes);
}

int b200_sixdof_set_schedule(b200_sixdof *h, uint64_t component_id, const void *rows, uint64_t bytes, uint64_t n_rows,
                             uint64_t first_tick)
{
    if (!h) return fail(B200_ERR_INVALID_ARGUMENT, "null handle");
    if (h->status != B200_OK) return fail(h->status, "handle is in a failed state");
    CU(h, cudaSetDevice(h->device));
    Column *c = h->find(component_id);
    if (!c) return fail(B200_ERR_COMPONENT_NOT_FOUND, "component not found: 0x%016llx", (unsigned long long)component_id);
    if (is_state_column(component_id))
        return fail(B200_ERR_INVALID_ARGUMENT, "column 0x%016llx is not an effector input: only effector input columns take a schedule",
                    (unsigned long long)component_id);
    if (h->graph_eff >= 0)
        return fail(B200_ERR_UNSUPPORTED, "input schedules are not supported on graph worlds (edge_fold gravity: small_world_kernel, "
                                          "nbody_tick_fused_kernel, graph_dense_world_kernel, the graph-force launch)");
    if (n_rows == 0) return fail(B200_ERR_INVALID_ARGUMENT, "an input schedule needs at least one row");
    const uint64_t row_bytes = column_bytes(h, *c);
    if (bytes != n_rows * row_bytes || (row_bytes && bytes / row_bytes != n_rows))
        return fail(B200_ERR_VALUE_SIZE_MISMATCH, "schedule of 0x%016llx: %llu rows of %llu bytes, got %llu bytes",
                    (unsigned long long)component_id, (unsigned long long)n_rows, (unsigned long long)row_bytes,
                    (unsigned long long)bytes);
    if (bytes && !rows) return fail(B200_ERR_INVALID_ARGUMENT, "null rows buffer");
    Schedule *old = h->find_schedule(component_id);
    int rc = B200_OK;
    if (old && (rc = materialise_schedule(h, *old))) return rc; // the column keeps the row the old schedule last used
    // device table: row r, plane p at table + (r*width + p)*ld, copied through the staging buffer a few rows at a time
    const uint64_t stride = (uint64_t)c->width * h->ld;
    double *table = nullptr;
    if (h->n_bodies) {
        if (cudaMalloc(&table, n_rows * stride * 8ull) != cudaSuccess) {
            (void)cudaGetLastError();
            return fail(B200_ERR_OUT_OF_MEMORY, "out of device memory for a schedule of %llu rows (%llu bytes)", (unsigned long long)n_rows,
                        (unsigned long long)(n_rows * stride * 8ull));
        }
        auto bail = [&](int code) { cudaFree(table); return code; };
        if (cudaMemsetAsync(table, 0, n_rows * stride * 8ull, h->stream) != cudaSuccess)
            return bail(cuda_fail(h, cudaGetLastError(), "cudaMemsetAsync(schedule)"));
        const uint64_t chunk_rows = std::max<uint64_t>(1, std::min<uint64_t>(n_rows, (64ull << 20) / row_bytes));
        if ((rc = ensure_staging(h, chunk_rows * row_bytes))) return bail(rc);
        for (uint64_t r0 = 0; r0 < n_rows; r0 += chunk_rows) {
            const uint64_t nr = std::min(chunk_rows, n_rows - r0);
            cudaError_t e = cudaMemcpyAsync(h->staging, (const char *)rows + r0 * row_bytes, nr * row_bytes, cudaMemcpyDefault, h->stream);
            for (uint64_t r = 0; r < nr && e == cudaSuccess; ++r) {
                e = launch_aos_to_soa(h->staging + r * (row_bytes / 8), table + (r0 + r) * stride, h->n_bodies, c->width, h->ld, h->stream);
                h->timings.kernel_launches++;
            }
            if (e != cudaSuccess) return bail(cuda_fail(h, e, "schedule upload"));
        }
        // the caller's buffer is only valid for this call, and the table an old schedule leaves may still be in use
        if (cudaStreamSynchronize(h->stream) != cudaSuccess) return bail(cuda_fail(h, cudaGetLastError(), "schedule upload sync"));
    }
    if (old) {
        if (old->table) cudaFree(old->table);
        old->table = table; old->n_rows = n_rows; old->first_tick = first_tick; old->pending = false;
    } else {
        Schedule s{};
        s.id = component_id; s.width = c->width; s.table = table; s.n_rows = n_rows; s.first_tick = first_tick;
        h->schedules.push_back(s);
    }
    return B200_OK;
}

int b200_sixdof_clear_schedule(b200_sixdof *h, uint64_t component_id)
{
    if (!h) return fail(B200_ERR_INVALID_ARGUMENT, "null handle");
    CU(h, cudaSetDevice(h->device));
    if (!h->find(component_id)) return fail(B200_ERR_COMPONENT_NOT_FOUND, "component not found: 0x%016llx", (unsigned long long)component_id);
    Schedule *s = h->find_schedule(component_id);
    if (!s) return B200_OK; // nothing bound: the column already drives its effector
    int rc = materialise_schedule(h, *s); // the column keeps the row its last tick used
    if (rc) return rc;
    CU(h, cudaStreamSynchronize(h->stream));
    if (s->table) cudaFree(s->table);
    h->schedules.erase(h->schedules.begin() + (s - h->schedules.data()));
    return B200_OK;
}

int b200_sixdof_step(b200_sixdof *h, uint64_t n_ticks)
{
    if (!h) return fail(B200_ERR_INVALID_ARGUMENT, "null handle");
    CU(h, cudaSetDevice(h->device));
    return do_step(h, n_ticks);
}

int b200_sixdof_sync(b200_sixdof *h)
{
    if (!h) return fail(B200_ERR_INVALID_ARGUMENT, "null handle");
    CU(h, cudaSetDevice(h->device));
    CU(h, cudaStreamSynchronize(h->stream));
    return B200_OK;
}

// Which input columns really have to cross PCIe: Force is cleared before any effector runs
// (clear_forces, six_dof.rs:148-150) so its input value is dead; WorldAccel only enters as
// `0 * a_prev` (rk4.rs:85-104), which FAST math does not evaluate.  EXACT keeps WorldAccel.
static bool input_is_live(const b200_sixdof *h, uint64_t id)
{
    if (id == B200_ID_FORCE) return false;
    if (id == B200_ID_WORLD_ACCEL) return h->desc.math_mode == B200_MATH_EXACT && h->desc.integrator == B200_INTEGRATOR_RK4;
    return true;
}

// Output columns the kernels never write (Inertia, effector input columns) are pass-through
// variables of the reference system (`builder.to_compiled_system()` returns every var): their
// output buffer is the input buffer's content, so it is filled host-to-host on worker threads
// while the PCIe link carries the columns that did change.
static bool output_is_pass_through(uint64_t id)
{
    return id != B200_ID_WORLD_POS && id != B200_ID_WORLD_VEL && id != B200_ID_WORLD_ACCEL && id != B200_ID_FORCE &&
           id != B200_ID_TICK && id != B200_ID_SIMULATION_TIME_STEP;
}

// Small batches (interactive single-vehicle sims: the reference's everyday case) are bound by the
// number of driver calls, not by bytes: pack every live input column into one pinned block, ONE
// host->device copy, ONE layout launch for all columns, the ticks, ONE layout launch, ONE copy back.
static int invoke_small(b200_sixdof *h, const uint8_t *const *in_cols, uint8_t *const *out_cols, uint64_t n_ticks)
{
    MultiColumns mi{}, mo{};
    uint64_t in_total = 0, out_total = 0;
    std::vector<std::pair<size_t, uint64_t>> in_map, out_map; // (column index, byte offset in the packed block)
    for (size_t i = 0; i < h->input_ids.size(); ++i) {
        Column *c = h->find(h->input_ids[i]);
        if (!in_cols[i]) continue; // not dirty: the device-resident copy stands
        if (c->global) { int rc = do_upload(h, c->id, in_cols[i], 8); if (rc) return rc; continue; }
        if (!input_is_live(h, c->id)) continue;
        mi.col[mi.n++] = {in_total, c->dev, c->width, 0};
        in_map.push_back({i, in_total * 8});
        in_total += h->n_bodies * c->width;
    }
    for (size_t i = 0; i < h->output_ids.size(); ++i) {
        Column *c = h->find(h->output_ids[i]);
        if (!out_cols[i] || c->global || output_is_pass_through(c->id)) continue;
        mo.col[mo.n++] = {out_total, c->dev, c->width, 0};
        out_map.push_back({i, out_total * 8});
        out_total += h->n_bodies * c->width;
    }
    const uint64_t need = std::max(in_total, out_total) * 8;
    if (h->host_pack_bytes < need) {
        if (h->host_pack) cudaFreeHost(h->host_pack);
        h->host_pack = nullptr; h->host_pack_bytes = 0;
        CU(h, cudaHostAlloc((void **)&h->host_pack, std::max<uint64_t>(need, 4096), cudaHostAllocDefault));
        h->host_pack_bytes = std::max<uint64_t>(need, 4096);
    }
    int rc = ensure_staging(h, std::max<uint64_t>(need, 8));
    if (rc) return rc;
    for (auto &m : in_map) {
        const Column *c = h->find(h->input_ids[m.first]);
        std::memcpy(h->host_pack + m.second, in_cols[m.first], h->n_bodies * c->width * 8);
    }
    mi.packed = mo.packed = h->staging;
    if (in_total) {
        CU(h, cudaMemcpyAsync(h->staging, h->host_pack, in_total * 8, cudaMemcpyHostToDevice, h->stream));
        CU(h, launch_multi_transpose(mi, h->n_bodies, h->ld, true, h->stream));
        h->timings.kernel_launches++;
    }
    rc = launch_ticks(h, 0, h->desc.n_worlds, n_ticks, h->stream);
    if (rc) return rc;
    commit_ping_pong(h, n_ticks);
    for (uint32_t k = 0; k < mo.n; ++k) mo.col[k].soa = h->find(h->output_ids[out_map[k].first])->dev; // after a ping-pong swap
    h->ticks_done += n_ticks;
    h->tick += n_ticks;
    h->timings.ticks += n_ticks;
    note_schedule_ticks(h, n_ticks);
    if (out_total) {
        CU(h, launch_multi_transpose(mo, h->n_bodies, h->ld, false, h->stream));
        h->timings.kernel_launches++;
        CU(h, cudaMemcpyAsync(h->host_pack, h->staging, out_total * 8, cudaMemcpyDeviceToHost, h->stream));
    }
    CU(h, cudaStreamSynchronize(h->stream));
    for (auto &m : out_map) {
        const Column *c = h->find(h->output_ids[m.first]);
        std::memcpy(out_cols[m.first], h->host_pack + m.second, h->n_bodies * c->width * 8);
    }
    for (size_t i = 0; i < h->output_ids.size(); ++i) {
        const Column *c = h->find(h->output_ids[i]);
        if (!out_cols[i]) continue;
        if (c->global) { rc = do_download(h, c->id, out_cols[i], 8); if (rc) return rc; continue; }
        if (!output_is_pass_through(c->id)) continue;
        bool filled = false;
        for (size_t k = 0; k < h->input_ids.size(); ++k)
            if (h->input_ids[k] == c->id && in_cols[k]) {
                if (in_cols[k] != out_cols[i]) std::memcpy(out_cols[i], in_cols[k], h->n_bodies * c->width * 8);
                filled = true;
            }
        if (!filled) { rc = do_download(h, c->id, out_cols[i], h->n_bodies * c->width * 8); if (rc) return rc; } // input was not dirty: the device copy is the value
    }
    h->timings.h2d_upload_ms = h->timings.kernel_invoke_ms = h->timings.d2h_download_ms = 0.0; // not separable here
    return B200_OK;
}

static int invoke_pipelined(b200_sixdof *h, const uint8_t *const *in_cols, uint8_t *const *out_cols, uint64_t n_ticks,
                            uint64_t worlds_per_chunk)
{
    const uint64_t N = h->desc.n_entities, M = h->desc.n_worlds;
    const uint64_t n_chunks = (M + worlds_per_chunk - 1) / worlds_per_chunk;
    if (!h->copy_in) {
        CU(h, cudaStreamCreateWithFlags(&h->copy_in, cudaStreamNonBlocking));
        CU(h, cudaStreamCreateWithFlags(&h->copy_out, cudaStreamNonBlocking));
    }
    // B200_PIPE_TRACE=1: per-range completion times of the three engines on stderr (diagnostic; timing events)
    static const bool trace = [] { const char *e = getenv("B200_PIPE_TRACE"); return e && atoi(e) != 0; }();
    std::vector<cudaEvent_t> trace_d2h;
    const auto host_t0 = std::chrono::steady_clock::now();
    auto host_ms = [&] { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - host_t0).count(); };
    double host_loop0 = 0.0, host_loop1 = 0.0;
    while (h->chunk_in.size() < n_chunks) {
        cudaEvent_t a, b;
        CU(h, cudaEventCreateWithFlags(&a, trace ? cudaEventDefault : cudaEventDisableTiming));
        CU(h, cudaEventCreateWithFlags(&b, trace ? cudaEventDefault : cudaEventDisableTiming));
        h->chunk_in.push_back(a);
        h->chunk_out.push_back(b);
    }
    // whole-batch AoS staging: column c of the inputs lives at in_off[c] (doubles)
    std::vector<uint64_t> in_off(h->input_ids.size(), 0), out_off(h->output_ids.size(), 0);
    uint64_t in_total = 0, out_total = 0;
    for (size_t i = 0; i < h->input_ids.size(); ++i) {
        const Column *c = h->find(h->input_ids[i]);
        in_off[i] = in_total;
        if (in_cols[i] && !c->global && input_is_live(h, c->id)) in_total += h->n_bodies * c->width;
    }
    for (size_t i = 0; i < h->output_ids.size(); ++i) {
        const Column *c = h->find(h->output_ids[i]);
        out_off[i] = out_total;
        if (out_cols[i] && !c->global && !output_is_pass_through(c->id)) out_total += h->n_bodies * c->width;
    }
    // host-to-host fill of the pass-through outputs, split over a few worker threads
    std::vector<size_t> late_downloads;
    std::vector<std::thread> fillers;
    struct Joiner { std::vector<std::thread> &v; ~Joiner() { for (auto &t : v) if (t.joinable()) t.join(); } } joiner{fillers};
    for (size_t i = 0; i < h->output_ids.size(); ++i) {
        const Column *c = h->find(h->output_ids[i]);
        if (!out_cols[i] || c->global || !output_is_pass_through(c->id)) continue;
        const uint8_t *src = nullptr;
        for (size_t k = 0; k < h->input_ids.size(); ++k) if (h->input_ids[k] == c->id) src = in_cols[k];
        if (!src) { late_downloads.push_back(i); continue; } // input not dirty: its value is the device-resident column
        if (src == out_cols[i]) continue;
        cudaPointerAttributes a_in{}, a_out{};
        const bool dev_in = cudaPointerGetAttributes(&a_in, src) == cudaSuccess && a_in.type == cudaMemoryTypeDevice;
        const bool dev_out = cudaPointerGetAttributes(&a_out, out_cols[i]) == cudaSuccess && a_out.type == cudaMemoryTypeDevice;
        (void)cudaGetLastError();
        const uint64_t bytes = h->n_bodies * c->width * 8ull;
        if (dev_in || dev_out) { // device-resident caller buffers: let the copy engine do it
            CU(h, cudaMemcpyAsync(out_cols[i], src, bytes, cudaMemcpyDefault, h->copy_out));
            continue;
        }
        const unsigned parts = bytes >= (8u << 20) ? 4u : 1u;
        for (unsigned t = 0; t < parts; ++t) {
            const uint64_t o0 = bytes * t / parts, o1 = bytes * (t + 1) / parts;
            uint8_t *dst = out_cols[i];
            fillers.emplace_back([dst, src, o0, o1] { std::memcpy(dst + o0, src + o0, o1 - o0); });
        }
    }
    if (h->stage_in_bytes < in_total * 8) {
        if (h->stage_in) CU(h, cudaFree(h->stage_in));
        h->stage_in = nullptr; h->stage_in_bytes = 0;
        CU(h, cudaMalloc(&h->stage_in, std::max<uint64_t>(in_total * 8, 8)));
        h->stage_in_bytes = in_total * 8;
    }
    if (h->stage_out_bytes < out_total * 8) {
        if (h->stage_out) CU(h, cudaFree(h->stage_out));
        h->stage_out = nullptr; h->stage_out_bytes = 0;
        CU(h, cudaMalloc(&h->stage_out, std::max<uint64_t>(out_total * 8, 8)));
        h->stage_out_bytes = out_total * 8;
    }
    // globals first (host-resident scalars)
    for (size_t i = 0; i < h->input_ids.size(); ++i) {
        const Column *c = h->find(h->input_ids[i]);
        if (c->global && in_cols[i]) { int rc = do_upload(h, c->id, in_cols[i], 8); if (rc) return rc; }
    }
    // the copy streams must not run ahead of work already queued on the compute stream
    CU(h, cudaEventRecord(h->ev[2], h->stream));
    CU(h, cudaStreamWaitEvent(h->copy_in, h->ev[2], 0));
    CU(h, cudaStreamWaitEvent(h->copy_out, h->ev[2], 0));
    CU(h, cudaEventRecord(h->ev[0], h->copy_in));

    host_loop0 = host_ms();
    for (uint64_t k = 0; k < n_chunks; ++k) {
        const uint64_t w0 = k * worlds_per_chunk, nw = std::min(worlds_per_chunk, M - w0);
        const uint64_t b0 = w0 * N, nb = nw * N;
        // H2D of this world range, every live input column (copy engine 1)
        for (size_t i = 0; i < h->input_ids.size(); ++i) {
            const Column *c = h->find(h->input_ids[i]);
            if (!in_cols[i] || c->global || !input_is_live(h, c->id)) continue;
            CU(h, cudaMemcpyAsync(h->stage_in + in_off[i] + b0 * c->width, (const double *)in_cols[i] + b0 * c->width,
                                  nb * c->width * 8, cudaMemcpyDefault, h->copy_in));
        }
        CU(h, cudaEventRecord(h->chunk_in[k], h->copy_in));
        if (k + 1 == n_chunks) CU(h, cudaEventRecord(h->ev[1], h->copy_in));
        // compute stream: AoS -> SoA, n ticks, SoA -> AoS
        CU(h, cudaStreamWaitEvent(h->stream, h->chunk_in[k], 0));
        for (size_t i = 0; i < h->input_ids.size(); ++i) {
            const Column *c = h->find(h->input_ids[i]);
            if (!in_cols[i] || c->global || !input_is_live(h, c->id)) continue;
            CU(h, launch_aos_to_soa(h->stage_in + in_off[i] + b0 * c->width, c->dev + b0, nb, c->width, h->ld, h->stream));
            h->timings.kernel_launches++;
        }
        int rc = launch_ticks(h, w0, nw, n_ticks, h->stream);
        if (rc) return rc;
        const bool flipped = h->nbody_fused && (n_ticks & 1); // live pose / velocity sit in the other plane set
        for (size_t i = 0; i < h->output_ids.size(); ++i) {
            const Column *c = h->find(h->output_ids[i]);
            if (!out_cols[i] || c->global || output_is_pass_through(c->id)) continue;
            const double *live = c->dev;
            if (flipped && c->id == B200_ID_WORLD_POS) live = h->pos_alt;
            if (flipped && c->id == B200_ID_WORLD_VEL) live = h->vel_alt;
            CU(h, launch_soa_to_aos(live + b0, h->stage_out + out_off[i] + b0 * c->width, nb, c->width, h->ld, h->stream));
            h->timings.kernel_launches++;
        }
        CU(h, cudaEventRecord(h->chunk_out[k], h->stream));
        if (k + 1 == n_chunks) CU(h, cudaEventRecord(h->ev[3], h->stream));
        // D2H of this world range (copy engine 2) overlaps the next range's H2D and ticks
        CU(h, cudaStreamWaitEvent(h->copy_out, h->chunk_out[k], 0));
        if (k == 0) CU(h, cudaEventRecord(h->ev[4], h->copy_out));
        for (size_t i = 0; i < h->output_ids.size(); ++i) {
            const Column *c = h->find(h->output_ids[i]);
            if (!out_cols[i] || c->global || output_is_pass_through(c->id)) continue;
            CU(h, cudaMemcpyAsync((double *)out_cols[i] + b0 * c->width, h->stage_out + out_off[i] + b0 * c->width,
                                  nb * c->width * 8, cudaMemcpyDefault, h->copy_out));
        }
        if (trace) {
            cudaEvent_t e;
            CU(h, cudaEventCreate(&e));
            CU(h, cudaEventRecord(e, h->copy_out));
            trace_d2h.push_back(e);
        }
    }
    host_loop1 = host_ms();
    commit_ping_pong(h, n_ticks);
    h->ticks_done += n_ticks;
    h->tick += n_ticks;
    h->timings.ticks += n_ticks;
    note_schedule_ticks(h, n_ticks);
    for (size_t i = 0; i < h->output_ids.size(); ++i) {
        const Column *c = h->find(h->output_ids[i]);
        if (c->global && out_cols[i]) { int rc = do_download(h, c->id, out_cols[i], 8); if (rc) return rc; }
    }
    CU(h, cudaEventRecord(h->ev[5], h->copy_out));
    CU(h, cudaStreamSynchronize(h->copy_out));
    CU(h, cudaStreamSynchronize(h->stream));
    CU(h, cudaStreamSynchronize(h->copy_in));
    for (size_t i : late_downloads) {
        const Column *c = h->find(h->output_ids[i]);
        int rc = do_download(h, c->id, out_cols[i], h->n_bodies * c->width * 8ull);
        if (rc) return rc;
    }
    if (trace) {
        fprintf(stderr, "[b200 pipe] host: enqueue loop %.3f..%.3f ms, synced at %.3f ms; device times from the first upload's start:\n",
                host_loop0, host_loop1, host_ms());
        for (uint64_t k = 0; k < n_chunks; ++k) {
            fprintf(stderr, "[b200 pipe]  range %2llu: upload done %.3f  ticks done %.3f  download done %.3f ms\n", (unsigned long long)k,
                    ev_ms(h->ev[0], h->chunk_in[k]), ev_ms(h->ev[0], h->chunk_out[k]), ev_ms(h->ev[0], trace_d2h[k]));
            cudaEventDestroy(trace_d2h[k]);
        }
    }
    // busy spans of the three engines; they overlap, so they do not add up to the call time
    h->timings.h2d_upload_ms = ev_ms(h->ev[0], h->ev[1]);
    h->timings.kernel_invoke_ms = ev_ms(h->ev[2], h->ev[3]);
    h->timings.d2h_download_ms = ev_ms(h->ev[4], h->ev[5]);
    return B200_OK;
}

int b200_sixdof_invoke_batch(b200_sixdof *h, const uint8_t *const *in_cols, uint8_t *const *out_cols, uint64_t n_ticks)
{
    if (!h) return fail(B200_ERR_INVALID_ARGUMENT, "null handle");
    if (!in_cols || !out_cols) return fail(B200_ERR_INVALID_ARGUMENT, "null column tables");
    if (h->status != B200_OK) return fail(h->status, "handle is in a failed state");
    CU(h, cudaSetDevice(h->device));
    // A NULL in_cols[i] means "not dirty" (World::dirty_components, world.rs:43,249-252): the device-resident copy of
    // that column stands.  A NULL out_cols[j] means the caller does not read that column after this batch.
    n_ticks = std::max<uint64_t>(n_ticks, 1); // `n.max(1)`, cranelift_exec.rs:135
    for (size_t i = 0; i < h->input_ids.size(); ++i)
        if (in_cols[i] && h->find_schedule(h->input_ids[i]))
            return fail(B200_ERR_INVALID_ARGUMENT, "input column 0x%016llx is driven by an input schedule: pass NULL for it",
                        (unsigned long long)h->input_ids[i]);

    // World ranges of ~kChunkBodies bodies: range k's PCIe download overlaps range k+1's upload
    // and ticks (two copy engines + the compute stream).  Small batches run as one range.
    static const uint64_t kEnvChunk = [] { const char *e = getenv("B200_CHUNK_BODIES"); return e ? (uint64_t)atoll(e) : (uint64_t)0; }();
    const uint64_t chunk_bodies = h->desc.invoke_chunk_bodies ? h->desc.invoke_chunk_bodies : (kEnvChunk ? kEnvChunk : 131072);
    const uint64_t N = std::max<uint64_t>(h->desc.n_entities, 1);
    uint64_t wpc = std::max<uint64_t>(1, chunk_bodies / N);
    if (N == 1 && wpc >= 128) wpc = wpc / 128 * 128;
    if (h->n_bodies == 0) wpc = std::max<uint64_t>(h->desc.n_worlds, 1);

    auto t0 = std::chrono::steady_clock::now();
    // host pointers only on the small path (it packs with memcpy); device-resident callers use the pipeline
    bool small = h->n_bodies > 0 && h->n_bodies * 32ull * 8ull <= (256ull << 10) && h->input_ids.size() <= 16 &&
                 !h->desc.invoke_chunk_bodies;
    if (small) { // the packed path memcpy()s: only for host-resident caller buffers
        for (size_t i = 0; i < h->input_ids.size() && small; ++i) {
            if (!in_cols[i] || h->find(h->input_ids[i])->global) continue;
            cudaPointerAttributes at{};
            if (cudaPointerGetAttributes(&at, in_cols[i]) == cudaSuccess && at.type == cudaMemoryTypeDevice) small = false;
        }
        for (size_t i = 0; i < h->output_ids.size() && small; ++i) {
            if (!out_cols[i] || h->find(h->output_ids[i])->global) continue;
            cudaPointerAttributes at{};
            if (cudaPointerGetAttributes(&at, out_cols[i]) == cudaSuccess && at.type == cudaMemoryTypeDevice) small = false;
        }
        (void)cudaGetLastError();
    }
    int rc = small ? invoke_small(h, in_cols, out_cols, n_ticks) : invoke_pipelined(h, in_cols, out_cols, n_ticks, wpc);
    if (rc) {
        // copies into the caller's buffers may still be queued: they must not outlive this call
        (void)cudaStreamSynchronize(h->stream);
        if (h->copy_in) (void)cudaStreamSynchronize(h->copy_in);
        if (h->copy_out) (void)cudaStreamSynchronize(h->copy_out);
        (void)cudaGetLastError();
        return rc;
    }
    h->timings.invoke_wall_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    return B200_OK;
}

int b200_sixdof_bind_tick(b200_sixdof *h)
{
    g_tick_handle = h;
    return B200_OK;
}

void b200_sixdof_tick(const uint8_t *const *in_cols, uint8_t **out_cols)
{
    b200_sixdof *h = g_tick_handle;
    if (!h) { fail(B200_ERR_INVALID_ARGUMENT, "b200_sixdof_tick: no handle bound on this thread"); return; }
    (void)b200_sixdof_invoke_batch(h, in_cols, out_cols, 1); // errors stay sticky on the handle / last_error
}

uint64_t b200_sixdof_trajectory_len(const b200_sixdof *h)
{
    if (!h || !h->traj || !h->desc.trajectory_every) return 0;
    return std::min<uint64_t>(h->ticks_done / h->desc.trajectory_every, h->desc.trajectory_capacity);
}

int b200_sixdof_trajectory_download(b200_sixdof *h, void *dst, uint64_t bytes)
{
    if (!h) return fail(B200_ERR_INVALID_ARGUMENT, "null handle");
    CU(h, cudaSetDevice(h->device));
    const uint64_t n = b200_sixdof_trajectory_len(h);
    const uint64_t W = h->traj_planes;
    const uint64_t want = n * h->n_bodies * W * 8ull;
    if (bytes != want) return fail(B200_ERR_VALUE_SIZE_MISMATCH, "trajectory is %llu bytes, got %llu", (unsigned long long)want, (unsigned long long)bytes);
    if (want == 0) return B200_OK;
    // convert in chunks through the staging buffer
    const uint64_t per_sample = h->n_bodies * W * 8ull;
    const uint64_t chunk = std::max<uint64_t>(1, std::min<uint64_t>(n, (256ull << 20) / per_sample));
    int rc = ensure_staging(h, chunk * per_sample);
    if (rc) return rc;
    for (uint64_t s0 = 0; s0 < n; s0 += chunk) {
        const uint64_t ns = std::min(chunk, n - s0);
        CU(h, launch_traj_to_aos(h->traj + s0 * W * h->ld, h->staging, ns, h->n_bodies, h->ld, (uint32_t)W, h->stream));
        h->timings.kernel_launches++;
        CU(h, cudaMemcpyAsync((char *)dst + s0 * per_sample, h->staging, ns * per_sample, cudaMemcpyDefault, h->stream));
        CU(h, cudaStreamSynchronize(h->stream));
    }
    return B200_OK;
}

uint32_t b200_sixdof_trajectory_width(const b200_sixdof *h) { return (h && h->traj) ? h->traj_planes : 0; }

int b200_sixdof_trajectory_reset(b200_sixdof *h)
{
    if (!h) return fail(B200_ERR_INVALID_ARGUMENT, "null handle");
    h->ticks_done = 0;
    return B200_OK;
}

uint64_t b200_sixdof_tick_count(const b200_sixdof *h) { return h ? h->tick : 0; }

int b200_sixdof_set_stream(b200_sixdof *h, void *cuda_stream, int use_own_stream)
{
    if (!h) return fail(B200_ERR_INVALID_ARGUMENT, "null handle");
    CU(h, cudaSetDevice(h->device));
    CU(h, cudaStreamSynchronize(h->stream));
    if (!use_own_stream) {
        if (h->own_stream && h->stream) cudaStreamDestroy(h->stream);
        h->stream = (cudaStream_t)cuda_stream;
        h->own_stream = false;
    } else if (!h->own_stream) {
        CU(h, cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
        h->own_stream = true;
    }
    return B200_OK;
}

int b200_sixdof_timings(const b200_sixdof *h, b200_timings *out)
{
    if (!h || !out) return fail(B200_ERR_INVALID_ARGUMENT, "null argument");
    *out = h->timings;
    return B200_OK;
}

int b200_sixdof_status(const b200_sixdof *h) { return h ? h->status : B200_ERR_INVALID_ARGUMENT; }

void *b200_sixdof_device_plane(b200_sixdof *h, uint64_t id, uint32_t plane)
{
    if (!h) return nullptr;
    Column *c = h->find(id);
    if (!c || c->global || plane >= c->width) return nullptr;
    return c->dev + (uint64_t)plane * h->ld;
}

uint64_t b200_sixdof_plane_stride(const b200_sixdof *h) { return h ? h->ld : 0; }

double b200_probe_copy_gbs(int device, uint64_t bytes, int iters)
{
    if (b200_device_count() <= 0) return -1.0;
    if (device >= 0 && cudaSetDevice(device) != cudaSuccess) return -1.0;
    void *a = nullptr, *b = nullptr;
    if (cudaMalloc(&a, bytes) != cudaSuccess || cudaMalloc(&b, bytes) != cudaSuccess) { cudaFree(a); (void)cudaGetLastError(); return -1.0; }
    cudaMemset(a, 1, bytes);
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    double best = 0.0;
    for (int i = 0; i < iters + 2; ++i) {
        cudaEventRecord(e0);
        cudaMemcpyAsync(b, a, bytes, cudaMemcpyDeviceToDevice);
        cudaEventRecord(e1);
        cudaEventSynchronize(e1);
        float ms = 0;
        cudaEventElapsedTime(&ms, e0, e1);
        if (i >= 2 && ms > 0) best = std::max(best, 2.0 * bytes / (ms * 1e-3) / 1e9);
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    cudaFree(a); cudaFree(b);
    return best;
}

// The EGM08 term stream the library builds at create (egm08_tables) for a degree-L coefficient pair: host-only, no GPU
// needed — lets a host (and tests/test_host_logic.py, against the oracle's tables) check what the kernel will read.
uint64_t b200_egm08_stream_len(uint32_t max_degree) { return 4ull * (max_degree + 1ull) * (max_degree + 2ull); }

int b200_egm08_stream(uint32_t max_degree, const double *c_bar, const double *s_bar, double *out, uint64_t out_len)
{
    if (!c_bar || !s_bar || !out) return fail(B200_ERR_INVALID_ARGUMENT, "null argument");
    if (max_degree > 128) return fail(B200_ERR_INVALID_ARGUMENT, "EGM08 max_degree must be 0..128 (got %u)", max_degree);
    if (out_len != b200_egm08_stream_len(max_degree))
        return fail(B200_ERR_VALUE_SIZE_MISMATCH, "the degree-%u stream holds %llu f64 (got %llu)", max_degree,
                    (unsigned long long)b200_egm08_stream_len(max_degree), (unsigned long long)out_len);
    const std::vector<double> t = egm08_tables((int)max_degree, c_bar, s_bar);
    std::memcpy(out, t.data(), t.size() * sizeof(double));
    return B200_OK;
}

// Self-test of the EXACT mode's shared-divisor divisions against div.rn.f64 (layout_kernels.cu:selftest_div_kernel):
// n_groups groups of four dividends over one divisor; out[0] = results that differ in any bit (must be 0),
// out[1] = groups answered without the __ddiv_rn fallback.
int b200_selftest_shared_divisor(int device, uint64_t seed, uint64_t n_groups, uint64_t *out)
{
    if (!out) return fail(B200_ERR_INVALID_ARGUMENT, "null argument");
    if (b200_device_count() <= 0) return B200_ERR_NO_DEVICE;
    if (device >= 0 && cudaSetDevice(device) != cudaSuccess) return cuda_fail(nullptr, cudaGetLastError(), "cudaSetDevice");
    unsigned long long *counts = nullptr, host[2] = {0, 0};
    if (cudaMalloc(&counts, sizeof host) != cudaSuccess) return cuda_fail(nullptr, cudaGetLastError(), "cudaMalloc(selftest)");
    cudaError_t e = cudaMemset(counts, 0, sizeof host);
    if (e == cudaSuccess) e = launch_selftest_div(seed, n_groups, counts, nullptr);
    if (e == cudaSuccess) e = cudaMemcpy(host, counts, sizeof host, cudaMemcpyDeviceToHost);
    cudaFree(counts);
    if (e != cudaSuccess) return cuda_fail(nullptr, e, "shared-divisor self-test");
    out[0] = host[0]; out[1] = host[1];
    return B200_OK;
}

double b200_probe_fp64_gflops(int device, int iters)
{
    if (b200_device_count() <= 0) return -1.0;
    if (device >= 0 && cudaSetDevice(device) != cudaSuccess) return -1.0;
    cudaDeviceProp prop{};
    int dev = 0;
    cudaGetDevice(&dev);
    cudaGetDeviceProperties(&prop, dev);
    const int blocks = prop.multiProcessorCount * 8;
    double *out = nullptr;
    if (cudaMalloc(&out, (size_t)blocks * 256 * 8) != cudaSuccess) return -1.0;
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    double best = 0.0;
    for (int i = 0; i < 5; ++i) {
        cudaEventRecord(e0);
        launch_probe_fp64(out, iters, blocks, nullptr);
        cudaEventRecord(e1);
        cudaEventSynchronize(e1);
        float ms = 0;
        cudaEventElapsedTime(&ms, e0, e1);
        if (i >= 1 && ms > 0) best = std::max(best, 2.0 * 8.0 * iters * blocks * 256.0 / (ms * 1e-3) / 1e9);
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    cudaFree(out);
    return best;
}

} // extern "C"
