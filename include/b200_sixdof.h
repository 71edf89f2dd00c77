/*
 * b200_sixdof.h — C ABI of the B200-native 6DOF rigid-body integrator.
 *
 * This library replaces, on the six_dof() hot path only, the executor seam of
 * elodin-sys/elodin's nox-py host:
 *
 *   enum WorldExec { Jax, Cranelift }            libs/nox-py/src/exec.rs:53-94
 *   CraneliftExec::invoke_batch(world, n, ..)    libs/nox-py/src/cranelift_exec.rs:129-195
 *   type TickFn = unsafe extern "C" fn(*const *const u8, *mut *mut u8)
 *                                                libs/nox-py/src/cranelift_exec.rs:11
 *   ExecMetadata{arg_ids, ret_ids, arg_slots}    libs/nox-py/src/exec.rs:18-29
 *
 * Everything below is plain C: opaque handle, POD descriptors, raw pointers and
 * sizes.  No C++/torch types cross the boundary; no exceptions cross it either
 * (every entry point returns an int status, 0 = ok, message via b200_last_error()).
 *
 * Data model (mirrors libs/nox-py/src/world.rs:25-29 `Column{buffer, entity_ids}`):
 *   a column is a dense little-endian f64 array [n_worlds][n_entities][width],
 *   row i of a world = i-th spawned entity that owns the component.  The
 *   reference has no world axis (one OS process per Monte-Carlo world,
 *   libs/monte-carlo/src/lib.rs:2083); n_worlds = 1 reproduces its layout
 *   byte for byte.  Columns are addressed by ComponentId = FNV-1a-64(name) with
 *   bit 63 cleared (libs/impeller2/src/types.rs:36-45).
 *
 * On the device every column is stored SoA: `width` planes of
 * n_worlds*n_entities doubles each (body index b = world*n_entities + entity).
 *
 * Threading: a handle is single-thread-affine, like the reference executor
 * ("moved once, never shared", cranelift_exec.rs:31-51).  One handle per GPU.
 */
#ifndef B200_SIXDOF_H
#define B200_SIXDOF_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200_SIXDOF_ABI_VERSION 3u

/* ---- status codes (0 = ok).  Names follow libs/nox-py/src/error.rs:7-44 ---- */
enum {
    B200_OK = 0,
    B200_ERR_COMPONENT_NOT_FOUND = 1, /* Error::ComponentNotFound            */
    B200_ERR_VALUE_SIZE_MISMATCH = 2, /* Error::ValueSizeMismatch            */
    B200_ERR_INVALID_ARGUMENT = 3,    /* Error::UnexpectedInput / MissingArg */
    B200_ERR_UNSUPPORTED = 4,         /* effector / integrator not built in  */
    B200_ERR_CUDA = 5,                /* Error::CraneliftBackend(String) analogue: backend failure (sticky per handle) */
    B200_ERR_NO_DEVICE = 6,           /* no CUDA device: there is NO CPU fallback */
    B200_ERR_OUT_OF_MEMORY = 7
};

/* ---- well-known component ids (FNV-1a-64 & ~(1<<63)); SURVEY §8a-7 ---- */
#define B200_ID_WORLD_ACCEL          0x019091805bc057f4ull
#define B200_ID_SIMULATION_TIME_STEP 0x08e7ddbb2cceaab5ull
#define B200_ID_TICK                 0x1e7683ef2ebc7684ull
#define B200_ID_WORLD_VEL            0x4b03b28a841edd5full
#define B200_ID_WORLD_POS            0x5d1c198a8e96e26eull
#define B200_ID_INERTIA              0x5fd14829c04c0f91ull
#define B200_ID_FORCE                0x675ad8afb3eeebe4ull

/* ---- integrators: libs/nox-py/src/integrator/{rk4,semi_implicit}.rs ---- */
enum {
    B200_INTEGRATOR_RK4 = 0,          /* Rk4::compile, rk4.rs:77-125 (incl. the v0-stage behaviour) */
    B200_INTEGRATOR_SEMI_IMPLICIT = 1 /* semi_implicit_euler, semi_implicit.rs:42-62 */
};

/* ---- arithmetic mode ---- */
enum {
    /* literal operation order of libs/nox/src/{spatial,quaternion}.rs, no FMA
     * contraction, IEEE div/sqrt: bit-identical to oracle/sixdof_oracle.c */
    B200_MATH_EXACT = 0,
    /* FMA contraction, hoisted reciprocals (hardware seed + 2 Newton steps), cross-product
     * rotations, R^-1/R cancelled around the mass divide, effectors folded once per launch;
     * agrees with EXACT to <= 1e-12 relative per tick (tests/test_parity_gpu.py states and
     * checks the tolerance).  Documented deviations from the literal arithmetic: the stage-1
     * term `0 * WorldAccel` (rk4.rs:85-104) is not evaluated, so a non-finite WorldAccel input
     * does not poison the step; denormal inputs to 1/x and 1/sqrt(x) flush to zero. */
    B200_MATH_FAST = 1
};

/* ---- trajectory ring contents (b200_sixdof_desc.trajectory_flags) ---- */
enum {
    /* a sample also carries WorldAccel[6] and Force[6] (the stage-4 values the tick leaves in the
     * ECS columns): 25 f64 per body instead of 13, i.e. every column `commit_world_head_unified`
     * (impeller2_server.rs:390-438) would have written for that telemetry tick */
    B200_TRAJ_FULL = 1
};

/* ---- built-in effectors (SURVEY §8a-12, §8a-8).  Evaluated in array order
 * inside every integrator stage on the stage state, accumulating into Force
 * after clear_forces (libs/nox-py/src/six_dof.rs:148-150,195). ---- */
enum {
    /* F.lin += g * m           examples/ball/sim.py:56-58, examples/rocket/main.py:292-294
     * p[0..2] = g */
    B200_EFF_GRAVITY_CONST = 1,
    /* quadratic drag on the stage velocity, examples/ball/sim.py:99-116
     * p[0] = Cd*rho, p[1] = area; column (optional) = wind (width 3), or wind + per-body
     * [Cd*rho, area] (width 5: Monte-Carlo worlds with their own drag parameters);
     * NOTE (reference behaviour): result torque is reset to 0. */
    B200_EFF_DRAG_QUADRATIC = 2,
    /* F.lin += (q @ axis) * thrust      examples/rocket/main.py:429-431
     * p[0..2] = body axis; column (width 1) = thrust per body */
    B200_EFF_THRUST_BODY = 3,
    /* F += q @ wrench (body -> world)   examples/rocket/main.py:407-413 (layout [tau,f])
     *                                   examples/falcon9/sim.py:659-672 (layout [f,tau], flag below)
     * column (width 6) = body-frame wrench per body */
    B200_EFF_WRENCH_BODY = 4,
    /* point-mass gravity + Coriolis + centrifugal in a rotating frame,
     * examples/falcon9/sim.py:350-361 + frames.py:91-109
     * p[0] = mu, p[1..3] = frame angular velocity */
    B200_EFF_GRAVITY_FRAME = 5,
    /* GraphQuery.edge_fold gravity, sequential fold per source body over its
     * out-edges in spawn order (libs/nox-py/src/graph.rs:177-236,
     * python/elodin/__init__.py:454-557); Force := fold(init 0).
     * NEWTON  : examples/three-body/main.py:63-70    p[0] = G
     * SOFTENED: examples/n-body/sim.py:349-361       p[0] = K^2, p[1] = softening */
    B200_EFF_GRAVITY_EDGES_NEWTON = 6,
    B200_EFF_GRAVITY_EDGES_SOFTENED = 7,
    /* F += column, a world-frame wrench [tau(3), f(3)] whose value is computed outside six_dof (a host system,
     * recorded telemetry): `force + SpatialForce(..)` of examples/cube-sat/main.py:516-527,
     * examples/drone/sim.py:99-103.  column (width 6). */
    B200_EFF_WRENCH_WORLD = 8,
    /* Reaction-wheel edge fold, examples/cube-sat/main.py:492-505: Force := fold over the body's K wheels (its
     * out-edges, spawn order) of SpatialForce(torque = q @ tau_k), init SpatialForce().  column (width 3K, K <= 8)
     * = the K wheel torques [tau_1 .. tau_K] of each body, body frame.  Like every edge_fold it OVERWRITES Force. */
    B200_EFF_TORQUE_BODY_FOLD = 9,
    /* point mass + J2 zonal gravity, libs/nox-py/python/elodin/j2.py:5-29 (J2.compute_field), applied as
     * force + SpatialForce(linear=field).  p[0] = mu, p[1] = J2, p[2] = r_ref */
    B200_EFF_GRAVITY_J2 = 10,
    /* spherical-harmonic gravity, libs/nox-py/python/elodin/egm08.py (EGM08.compute_field), applied as
     * force + SpatialForce(linear=field) (examples/cube-sat/main.py:516-527).  p[0] = mu, p[1] = r_ref, p[2] = max_degree L
     * (<= 128); table0 / table1 = the fully normalised C / S coefficients, [(L+1)][(L+1)] f64 row-major (row = degree) —
     * what the reference loads from C_normal.npy / S_normal.npy (a run-time download, so no golden pins it: with C20
     * alone the field equals GRAVITY_J2's to rounding).  Both math modes evaluate it with the oracle's operation order. */
    B200_EFF_GRAVITY_EGM08 = 11
};

#define B200_EFF_FLAG_WRENCH_LINEAR_FIRST 1u /* wrench column is [f(3), tau(3)] (falcon9) */

#define B200_MAX_EFFECTORS 8u

typedef struct b200_effector {
    uint32_t kind;          /* B200_EFF_*                                           */
    uint32_t flags;         /* B200_EFF_FLAG_*                                      */
    double   p[8];          /* constants, meaning per kind                          */
    uint64_t column_id;     /* ComponentId of the per-body input column, 0 = none   */
    uint32_t column_width;  /* f64 per body in that column                          */
    uint32_t reserved;
    uint64_t n_edges;       /* GRAVITY_EDGES_*: directed edges, spawn order         */
    const uint32_t *edge_from; /* entity row index within a world                   */
    const uint32_t *edge_to;
    const uint8_t *entity_mask; /* [n_entities] or NULL: 1 = the effector applies to that entity row.
                                   Mirrors the reference's query join (query.rs:672-710): an @el.map
                                   effector only runs on entities that own every component it reads
                                   (e.g. drag only on bodies with a `wind` component).  Copied at create. */
    const double *table0;       /* ABI v3.  GRAVITY_EGM08: C coefficients; copied at create; NULL otherwise  */
    const double *table1;       /*          GRAVITY_EGM08: S coefficients                                     */
    uint64_t table_len;         /*          (L+1)^2                                                            */
} b200_effector;

typedef struct b200_sixdof_desc {
    uint32_t abi_version;      /* B200_SIXDOF_ABI_VERSION                            */
    uint32_t integrator;       /* B200_INTEGRATOR_*                                  */
    uint32_t math_mode;        /* B200_MATH_*                                        */
    uint32_t n_effectors;      /* <= B200_MAX_EFFECTORS                              */
    uint64_t n_entities;       /* bodies per world (rows of every Body column)       */
    uint64_t n_worlds;         /* Monte-Carlo world batch (>= 1)                     */
    double   sim_time_step;    /* SimulationTimeStep component (globals.rs:9); stage dt, rk4.rs:90 */
    double   time_step;        /* six_dof(time_step=..) override of the final combine dt (rk4.rs:83);
                                  NaN = none (use sim_time_step)                      */
    const b200_effector *effectors;
    int32_t  device;           /* CUDA ordinal, -1 = current device                  */
    uint32_t max_fused_ticks;  /* ticks one launch may keep in registers (0/1 = one tick per launch);
                                  only used when no effector couples bodies          */
    uint32_t trajectory_every; /* 0 = off; k = record (pos,vel) every k ticks         */
    uint32_t invoke_chunk_bodies; /* b200_sixdof_invoke_batch splits the world axis into ranges of about
                                  this many bodies so that range k's download overlaps range k+1's
                                  upload and ticks; 0 = default (131072)                */
    uint64_t trajectory_capacity; /* samples the device ring can hold                 */
    uint32_t trajectory_flags; /* B200_TRAJ_*                                        */
    uint32_t reserved0;        /* must be 0                                          */
} b200_sixdof_desc;

typedef struct b200_timings {  /* TickTimings analogue, libs/nox-py/src/profile.rs — of the last
                                  invoke_batch: busy spans of the upload copy engine, the compute stream
                                  and the download copy engine (they overlap) and the call's wall time */
    double h2d_upload_ms;
    double kernel_invoke_ms;
    double d2h_download_ms;
    double invoke_wall_ms;
    uint64_t kernel_launches;  /* launches of this library's kernels since create   */
    uint64_t ticks;            /* ticks integrated since create                      */
} b200_timings;

typedef struct b200_sixdof b200_sixdof; /* opaque */

/* FNV-1a-64(name) & ~(1<<63): ComponentId::new, libs/impeller2/src/types.rs:40-45 */
uint64_t b200_component_id(const char *name);

/* thread-local message of the last failing call (never NULL) */
const char *b200_last_error(void);

/* number of visible CUDA devices, or a negative status; never falls back to CPU */
int b200_device_count(void);

/* Page-locked host memory for column buffers (optional: any host pointer works,
 * pinned ones copy at full PCIe speed and asynchronously). */
void *b200_host_alloc(uint64_t bytes);
/* ... on the NUMA node of `device`'s PCIe root (-1 = current device): mmap + mbind + cudaHostRegister; falls back to
 * b200_host_alloc when the node is unknown.  With 4 GPUs per socket the host memory system, not PCIe, bounds the
 * columns' round trip unless every rank's buffers are node-local. */
void *b200_host_alloc_local(uint64_t bytes, int device);
void b200_host_free(void *p); /* either kind */
/* diagnostics: NUMA node of a GPU's PCIe root / of the first page of a host buffer; -1 = unknown */
int b200_device_numa_node(int device);
int b200_host_node_of(const void *p);

/* Build an executor for one world batch.  Replaces CraneliftExec::new
 * (cranelift_exec.rs:54-127): allocates device-resident SoA columns and the
 * output tables.  All columns start zeroed except inertia-independent defaults;
 * callers upload initial state with b200_sixdof_upload / _invoke_batch. */
int b200_sixdof_create(const b200_sixdof_desc *desc, b200_sixdof **out);
void b200_sixdof_destroy(b200_sixdof *h);

/* ExecMetadata.arg_ids / ret_ids (exec.rs:18-29).  Inputs in first-init order,
 * outputs sorted by ComponentId (BTreeMap order) — SURVEY §8a-7.  Returns the
 * count; writes at most `cap` ids. */
uint32_t b200_sixdof_input_ids(const b200_sixdof *h, uint64_t *ids, uint32_t cap);
uint32_t b200_sixdof_output_ids(const b200_sixdof *h, uint64_t *ids, uint32_t cap);
/* byte length of a column's host buffer (n_worlds*n_entities*width*8; 8 for the
 * two globals), 0 if the handle has no such column */
uint64_t b200_sixdof_column_bytes(const b200_sixdof *h, uint64_t component_id);

/* Host (or device: the copy direction is inferred, cudaMemcpyDefault) AoS column
 * -> device SoA planes, and back.  `bytes` must equal b200_sixdof_column_bytes
 * (else B200_ERR_VALUE_SIZE_MISMATCH, as cranelift_exec.rs:175-177,188-190). */
int b200_sixdof_upload(b200_sixdof *h, uint64_t component_id, const void *src, uint64_t bytes);
int b200_sixdof_download(b200_sixdof *h, uint64_t component_id, void *dst, uint64_t bytes);

/* Input schedules: drive an effector input column from a table of per-tick rows held on the device, so that a
 * thrust curve, a recorded input or a per-world open-loop profile runs in fused, device-resident launches.
 *   rows        n_rows rows, each in the column's host layout [n_worlds][n_entities][width] f64, so
 *               bytes == n_rows * b200_sixdof_column_bytes (else B200_ERR_VALUE_SIZE_MISMATCH).  Copied at this call.
 *   row rule    the tick whose Tick column value is k reads row clamp(k - first_tick, 0, n_rows - 1): the first row
 *               before the table starts, the last one after it ends.  k is the Tick value (invoke_batch: the `tick`
 *               input it is handed), not the trajectory tick count a trajectory reset restarts.
 *   readback    after ticks, the column (download, invoke_batch output) reads back as the row its last tick used.
 *   inputs      invoke_batch refuses a non-NULL input for a scheduled column, and upload refuses the column
 *               (B200_ERR_INVALID_ARGUMENT): the schedule owns it.
 * Only effector input columns take a schedule (state columns and the globals: B200_ERR_INVALID_ARGUMENT).  Graph
 * worlds (an edge_fold gravity effector) are B200_ERR_UNSUPPORTED, as is b200_sixdof_step_row_sharded while a
 * schedule is bound.  Setting a scheduled column again replaces its schedule.  Clearing leaves the column holding its
 * last-used row; later ticks read the column again.  The table takes n_rows * width * plane stride * 8 bytes of
 * device memory (B200_ERR_OUT_OF_MEMORY if that fails). */
int b200_sixdof_set_schedule(b200_sixdof *h, uint64_t component_id, const void *rows, uint64_t bytes, uint64_t n_rows,
                             uint64_t first_tick);
int b200_sixdof_clear_schedule(b200_sixdof *h, uint64_t component_id);

/* Advance the device-resident world n_ticks (asynchronous on the handle's
 * stream).  tick += n_ticks. */
int b200_sixdof_step(b200_sixdof *h, uint64_t n_ticks);
int b200_sixdof_sync(b200_sixdof *h);

/* The reference-shaped call: CraneliftExec::invoke_batch (cranelift_exec.rs:129-195).
 * in_cols[i]  = host buffer of input_ids[i]  (borrowed for the call only)
 * out_cols[j] = host buffer of output_ids[j] (caller-owned, never aliasing an input)
 * Uploads every input column, integrates max(n_ticks,1) ticks on the device,
 * downloads every output column, synchronises.
 * Because the state is device-resident between calls, two entries may be NULL:
 *   in_cols[i]  == NULL: the column is not dirty — the host has not modified it since the previous call
 *                        (World::dirty_components, libs/nox-py/src/world.rs:43,249-252) — the device copy stands;
 *   out_cols[j] == NULL: the caller does not read that column after this batch (e.g. WorldAccel / Force between
 *                        telemetry cycles, pass-through Inertia): it is neither downloaded nor filled. */
int b200_sixdof_invoke_batch(b200_sixdof *h, const uint8_t *const *in_cols,
                             uint8_t *const *out_cols, uint64_t n_ticks);

/* TickFn-shaped shim (cranelift_exec.rs:11): one tick, bound to a thread-local
 * handle.  Returns void like the reference; errors are sticky on the handle. */
int b200_sixdof_bind_tick(b200_sixdof *h);
void b200_sixdof_tick(const uint8_t *const *in_cols, uint8_t **out_cols);

/* Trajectory ring: samples of (world_pos[7], world_vel[6]) — with B200_TRAJ_FULL also
 * (world_accel[6], force[6]) — taken every `trajectory_every` ticks.  Download layout
 * [samples][n_worlds][n_entities][width], width = b200_sixdof_trajectory_width() = 13 | 25.
 * The ring lets a telemetry_rate < simulation_rate run stay device-resident between samples:
 * upload once, step, read the samples back in one transfer. */
uint64_t b200_sixdof_trajectory_len(const b200_sixdof *h);
uint32_t b200_sixdof_trajectory_width(const b200_sixdof *h);
int b200_sixdof_trajectory_download(b200_sixdof *h, void *dst, uint64_t bytes);
int b200_sixdof_trajectory_reset(b200_sixdof *h);

/* plumbing */
uint64_t b200_sixdof_tick_count(const b200_sixdof *h);
/* Run the handle's work on a caller-owned cudaStream_t (`cuda_stream`, where NULL is
 * the legacy default stream, e.g. torch.cuda.current_stream().cuda_stream), or, with
 * use_own_stream != 0, go back to the handle's private non-blocking stream. */
int b200_sixdof_set_stream(b200_sixdof *h, void *cuda_stream, int use_own_stream);
int b200_sixdof_timings(const b200_sixdof *h, b200_timings *out);
int b200_sixdof_status(const b200_sixdof *h);                  /* sticky status of the handle */
/* raw device plane pointer (plane p of a column), for zero-copy interop (NCCL gather) */
void *b200_sixdof_device_plane(b200_sixdof *h, uint64_t component_id, uint32_t plane);
uint64_t b200_sixdof_plane_stride(const b200_sixdof *h); /* doubles between planes */

/* ---- multi-GPU (SURVEY §8e).  Worlds shard across GPUs — one handle per GPU, one process (or thread) per
 * handle, no data-path collective — exactly like the reference's one-OS-process-per-world Monte-Carlo driver
 * (libs/monte-carlo/src/lib.rs:2083).  The one exchange is the end-of-run gather of the trajectory ring, over
 * NCCL (NVLink 5 / NVSwitch).  NCCL is bound at run time (dlopen of libnccl.so.2: the copy the host process already
 * loaded, else the system one); b200_comm_available() == 0 means it could not be found. ---- */
#define B200_COMM_ID_BYTES 128u                      /* sizeof(ncclUniqueId) */
typedef struct b200_comm b200_comm;                   /* opaque: one NCCL communicator rank */
int b200_comm_available(void);
int b200_comm_version(void);                          /* NCCL version code, 0 if unavailable */
/* rank 0 creates the id and hands its bytes to every rank over any channel the host has (the reference's
 * Monte-Carlo driver would put it in context.json); then every rank calls b200_comm_create. */
int b200_comm_unique_id(uint8_t *out, uint32_t bytes);
int b200_comm_create(const uint8_t *id, int n_ranks, int rank, int device, b200_comm **out);
void b200_comm_destroy(b200_comm *c);
int b200_comm_rank(const b200_comm *c);
int b200_comm_size(const b200_comm *c);
double b200_comm_last_ms(const b200_comm *c);         /* device time of the last gather (layout kernel + collective) */
/* World-sharded all-gather of the trajectory ring.  Rank r holds worlds_per_rank[r] worlds (same samples, entities
 * and ring width everywhere; ragged world counts allowed).  On return `dst` (device or host memory) holds
 * [sum(worlds)][samples][n_entities][width] f64 in rank order on every rank; dst_bytes must equal
 * b200_sixdof_trajectory_gather_bytes(). */
uint64_t b200_sixdof_trajectory_gather_bytes(const b200_sixdof *h, const uint64_t *worlds_per_rank, int n_ranks);
int b200_sixdof_trajectory_allgather(b200_sixdof *h, b200_comm *c, const uint64_t *worlds_per_rank, void *dst,
                                     uint64_t dst_bytes);

/* ONE world, source rows split over the ranks (SURVEY §8e second case; needs dense edge_fold gravity, n_worlds = 1,
 * n_entities divisible by the rank count).  Every rank creates the same handle and uploads the same initial state,
 * then calls this instead of b200_sixdof_step: per tick it folds and integrates its own rows and all-gathers the
 * rows' new position / velocity planes over NCCL; after the call every rank holds the complete world.
 * At N = 1024 replicas (every GPU integrates the whole world, no exchange) are faster — the tick is a ~10 us
 * latency chain and the exchange adds to it; row shards pay off for worlds of several thousand bodies
 * (DESIGN.md §7, measured by bench.py `multi_gpu.nbody_1024_single_world`). */
int b200_sixdof_step_row_sharded(b200_sixdof *h, b200_comm *c, uint64_t n_ticks);

/* Peer window for the row-sharded world: compute and exchange without a collective in the tick loop.  Every rank
 * allocates a window (the x, v planes of the whole world, twice — tick-count parity — plus one delivery counter per
 * rank), the ranks swap the windows' CUDA IPC handles through the communicator and map each other's.  With a window
 * attached, b200_sixdof_step_row_sharded runs per tick: wait until every rank's rows of this tick count have landed
 * here -> gravity from the window -> integrate own rows -> store the rows' new x, v straight into every rank's window
 * over NVLink and release each counter.  Only the call's last tick still all-gathers (attitude, WorldAccel, Force of
 * the other ranks' rows).  Results are bit-identical to the NCCL route and to replicas.
 * Collective: every rank of `c` calls attach (and detach / b200_comm_destroy) with handles of the same shape; one
 * window per communicator.  Returns B200_ERR_UNSUPPORTED on every rank if any rank cannot map the windows (no IPC
 * between the processes) — the NCCL route keeps working.  B200_ROW_PEER=0 ignores an attached window. */
#define B200_MAX_PEERS 16
int b200_comm_peer_attach(b200_comm *c, b200_sixdof *h);
int b200_comm_peer_attached(const b200_comm *c);
void b200_comm_peer_detach(b200_comm *c);

/* Concurrent host<->device copy bandwidth of one GPU through pinned `host` (>= h2d_bytes + d2h_bytes): out[0] = H2D
 * GB/s, out[1] = D2H GB/s, both directions running at once — the ceiling an invoke_batch round trip sits under. */
int b200_probe_pcie_gbs(int device, void *host, uint64_t h2d_bytes, uint64_t d2h_bytes, int iters, double *out);
/* The same with kernels instead of the copy engines (SMs reading / writing mapped pinned host memory, `blocks` CTAs of
 * 256 threads per direction): B200_ERR_UNSUPPORTED when `host` is not mapped into the device address space. */
int b200_probe_zero_copy_gbs(int device, void *host, uint64_t h2d_bytes, uint64_t d2h_bytes, int iters, int blocks, double *out);

/* FP64 / HBM probes used by bench.py to report the roofs next to the kernel
 * numbers (device-timed, returns GB/s resp. GFLOP/s, <0 on error) */
double b200_probe_copy_gbs(int device, uint64_t bytes, int iters);
double b200_probe_fp64_gflops(int device, int iters);
/* The term stream a GRAVITY_EGM08 effector of this degree is evaluated from (DESIGN.md §5): eight f64 per (m, l) term in
 * consumption order — recursion constants of A at (l, m) and of B at (l+1, m+1), C, S, nq1, nq2.  Host-only. */
uint64_t b200_egm08_stream_len(uint32_t max_degree);
int b200_egm08_stream(uint32_t max_degree, const double *c_bar, const double *s_bar, double *out, uint64_t out_len);
/* Self-test of the EXACT mode's division-by-a-shared-divisor route (sixdof_device.cuh ex::div_rcp) against the GPU's
 * IEEE division on n_groups pseudo-random operand groups covering every encoding class: out[0] = results differing
 * in any bit (0 on a correct build), out[1] = groups that did not need the __ddiv_rn fallback. */
int b200_selftest_shared_divisor(int device, uint64_t seed, uint64_t n_groups, uint64_t *out);

#ifdef __cplusplus
}
#endif
#endif /* B200_SIXDOF_H */
