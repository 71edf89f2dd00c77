// Multi-GPU plumbing of libb200_sixdof behind the C ABI (include/b200_sixdof.h, "multi-GPU" section).
//
// Worlds shard across GPUs with no data-path collective (SURVEY §8e); the one exchange the path has is the
// end-of-run gather of the device trajectory ring.  It runs over NCCL (NVLink 5 / NVSwitch), which this library
// binds at run time: dlopen("libnccl.so.2") — the copy a host process already loaded (e.g. torch's) if there is
// one, the system one otherwise — so libb200_sixdof.so itself links nothing but the CUDA runtime and a host
// that never gathers never needs NCCL installed.
#include <dlfcn.h>

#include <algorithm>
#include <cstring>
#include <mutex>
#include <vector>

#include <nccl.h> // types and prototypes only; every call goes through the table below

#include "sixdof_handle.h"
#include "sixdof_launch.h"

using namespace b200;

namespace {

struct NcclApi {
    void *lib = nullptr;
    decltype(&ncclGetUniqueId) GetUniqueId = nullptr;
    decltype(&ncclCommInitRank) CommInitRank = nullptr;
    decltype(&ncclCommDestroy) CommDestroy = nullptr;
    decltype(&ncclGetErrorString) GetErrorString = nullptr;
    decltype(&ncclBroadcast) Broadcast = nullptr;
    decltype(&ncclAllGather) AllGather = nullptr;
    decltype(&ncclGroupStart) GroupStart = nullptr;
    decltype(&ncclGroupEnd) GroupEnd = nullptr;
    decltype(&ncclGetVersion) GetVersion = nullptr;
    bool ok = false;
};

NcclApi &nccl()
{
    static NcclApi api;
    static std::once_flag once;
    std::call_once(once, [] {
        void *lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD | RTLD_GLOBAL); // the host process's copy, if any
        if (!lib) lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
        if (!lib) lib = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
        if (!lib) return;
        api.lib = lib;
#define SYM(name) api.name = reinterpret_cast<decltype(api.name)>(dlsym(lib, "nccl" #name))
        SYM(GetUniqueId); SYM(CommInitRank); SYM(CommDestroy); SYM(GetErrorString); SYM(Broadcast); SYM(AllGather);
        SYM(GroupStart); SYM(GroupEnd); SYM(GetVersion);
#undef SYM
        api.ok = api.GetUniqueId && api.CommInitRank && api.CommDestroy && api.GetErrorString && api.Broadcast &&
                 api.AllGather && api.GroupStart && api.GroupEnd;
    });
    return api;
}

int nccl_fail(ncclResult_t r, const char *what)
{
    return fail(B200_ERR_CUDA, "NCCL error in %s: %s", what, nccl().GetErrorString ? nccl().GetErrorString(r) : "?");
}

#define NC(call)                                             \
    do {                                                     \
        ncclResult_t r_ = (call);                            \
        if (r_ != ncclSuccess) return nccl_fail(r_, #call);  \
    } while (0)

} // namespace

struct b200_comm {
    ncclComm_t comm = nullptr;
    int n_ranks = 1, rank = 0, device = 0;
    double *send = nullptr, *recv = nullptr; // device staging of the gather
    uint64_t send_bytes = 0, recv_bytes = 0;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    double last_ms = 0.0;
    // peer window of the row-sharded world (b200_comm_peer_attach): one allocation per rank, mapped into every
    // other rank's address space through CUDA IPC, written over NVLink by the producing GPU
    struct Window {
        const b200_sixdof *owner = nullptr;
        uint64_t owner_serial = 0, ld = 0;     // the handle the window was sized for (address + creation serial)
        double *base[B200_MAX_PEERS] = {};  // rank r's window as mapped here ([rank] = the local allocation)
        unsigned *ctr = nullptr;            // block counter of the push kernel (local)
    } win;
};

// Layout of a peer window: X[2][6][ld] doubles (parity of the tick count; planes x y z vx vy vz of every row of
// the world), then B200_MAX_PEERS uint64 delivery counters: flags[r] = ticks whose rows rank r has delivered here.
static inline uint64_t win_doubles(uint64_t ld) { return 2ull * 6ull * ld; }
static inline size_t win_bytes(uint64_t ld) { return (size_t)(win_doubles(ld) * 8ull + B200_MAX_PEERS * 8ull + 64); }

namespace b200 {

// trajectory ring (SoA: sample s, plane p at traj + (s*W + p)*ld) -> world-major rows
//   out[((world*S + s)*N + entity)*W + p]
// so that a rank's worlds are one contiguous block of the world-sharded result.
static constexpr int kGTile = 128;
__global__ void __launch_bounds__(kGTile) traj_world_major_kernel(const double *__restrict__ traj, double *__restrict__ out,
                                                                  uint64_t n_bodies, uint32_t n_entities, uint32_t W, uint64_t S,
                                                                  uint64_t ld)
{
    extern __shared__ double tile[]; // kGTile * (W | 1)
    const uint32_t pitch = W | 1u;
    const uint64_t base = (uint64_t)blockIdx.x * kGTile, s = blockIdx.y;
    const uint32_t nb = (uint32_t)min((uint64_t)kGTile, n_bodies - base);
    const double *src = traj + s * (uint64_t)W * ld;
    if (threadIdx.x < nb)
        for (uint32_t k = 0; k < W; ++k) tile[threadIdx.x * pitch + k] = src[(uint64_t)k * ld + base + threadIdx.x];
    __syncthreads();
    for (uint32_t i = threadIdx.x; i < nb * W; i += kGTile) {
        const uint32_t r = i / W, k = i - r * W;
        const uint64_t b = base + r, world = b / n_entities, ent = b - world * n_entities;
        out[((world * S + s) * n_entities + ent) * W + k] = tile[r * pitch + k];
    }
}

// ------------------------------------------------------------------ peer-window kernels (row-sharded world)

// X[par] <- the linear position / velocity planes of the whole local world; flags[r] = max(flags[r], T)
__global__ void __launch_bounds__(256) peer_fill_kernel(const double *__restrict__ pos, const double *__restrict__ vel,
                                                        double *__restrict__ X, unsigned long long *flags, uint64_t ld,
                                                        uint32_t n, int n_ranks, unsigned long long T)
{
    const uint32_t i = blockIdx.x * 256u + threadIdx.x;
    if (i < n) {
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            X[(uint64_t)k * ld + i] = pos[(uint64_t)(4 + k) * ld + i];
            X[(uint64_t)(3 + k) * ld + i] = vel[(uint64_t)(3 + k) * ld + i];
        }
    }
    if (blockIdx.x == 0 && threadIdx.x < (unsigned)n_ranks) atomicMax(flags + threadIdx.x, T); // a faster peer may already be one ahead
}

// Spins until rank r has delivered the rows of tick count `need` into this GPU's window.
__device__ __forceinline__ void peer_wait_one(const unsigned long long *flag, unsigned long long need)
{
    unsigned long long t0, now, v;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
    for (;;) {
        asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(flag) : "memory");
        if (v >= need) return;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
        if (now - t0 > 20000000000ull) __trap(); // 20 s without the peer's rows: fail the handle instead of hanging the GPU
        __nanosleep(64);
    }
}

// Holds the stream until every rank's rows of tick count `need` are here (first tick of a call; later ticks wait at
// the end of the previous tick's push kernel).
__global__ void peer_wait_kernel(const unsigned long long *flags, int n_ranks, unsigned long long need)
{
    if (threadIdx.x < (unsigned)n_ranks) peer_wait_one(flags + threadIdx.x, need);
}

struct PeerPush {
    const double *pos, *vel;      // local planes, already shifted to this rank's first row
    double *dst[B200_MAX_PEERS];  // X[next parity] of every rank, shifted to this rank's first row
    unsigned long long *flag[B200_MAX_PEERS]; // &flags_r[me]
    unsigned *ctr;
    const unsigned long long *wait; // local delivery counters, or nullptr: do not wait for the peers' rows of `value`
    uint64_t ld_src, ld_dst;
    uint32_t rows;
    int n_ranks;
    unsigned long long value;     // tick count the rows belong to
};

// This rank's new rows -> every rank's window (NVLink stores), then one release per peer once every block is through;
// the same block then waits for the peers' rows of the same tick count, so the next tick's gravity launches straight
// behind this kernel.
__global__ void __launch_bounds__(128) peer_push_kernel(const __grid_constant__ PeerPush a)
{
    const uint32_t i = blockIdx.x * 128u + threadIdx.x, k = blockIdx.y; // plane k of x y z vx vy vz
    if (i < a.rows) {
        const double v = k < 3 ? a.pos[(uint64_t)(4 + k) * a.ld_src + i] : a.vel[(uint64_t)k * a.ld_src + i];
        for (int r = 0; r < a.n_ranks; ++r) a.dst[r][(uint64_t)k * a.ld_dst + i] = v;
    }
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned total = gridDim.x * gridDim.y;
        if (atomicAdd(a.ctr, 1u) == total - 1u) {
            *a.ctr = 0u;
            __threadfence_system();
            for (int r = 0; r < a.n_ranks; ++r)
                asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(a.flag[r]), "l"(a.value) : "memory");
            if (a.wait)
                for (int r = 0; r < a.n_ranks; ++r) peer_wait_one(a.wait + r, a.value);
        }
    }
}

// plain grid-stride copy of 16-byte words: the PCIe probe's SM-driven leg (one side is mapped pinned host memory)
__global__ void __launch_bounds__(256) copy16_kernel(const double2 *__restrict__ src, double2 *__restrict__ dst, uint64_t n)
{
    for (uint64_t i = (uint64_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (uint64_t)gridDim.x * 256) dst[i] = src[i];
}

} // namespace b200

extern "C" {

int b200_comm_available(void) { return nccl().ok ? 1 : 0; }

int b200_comm_version(void)
{
    int v = 0;
    if (nccl().ok && nccl().GetVersion) nccl().GetVersion(&v);
    return v;
}

int b200_comm_unique_id(uint8_t *out, uint32_t bytes)
{
    if (!out || bytes < B200_COMM_ID_BYTES) return fail(B200_ERR_INVALID_ARGUMENT, "unique id buffer must hold %u bytes", B200_COMM_ID_BYTES);
    if (!nccl().ok) return fail(B200_ERR_UNSUPPORTED, "libnccl.so.2 could not be loaded: %s", dlerror() ? dlerror() : "not found");
    static_assert(sizeof(ncclUniqueId) == B200_COMM_ID_BYTES, "NCCL unique id size");
    ncclUniqueId id;
    NC(nccl().GetUniqueId(&id));
    std::memcpy(out, &id, sizeof id);
    return B200_OK;
}

int b200_comm_create(const uint8_t *id_bytes, int n_ranks, int rank, int device, b200_comm **out)
{
    if (!id_bytes || !out || n_ranks < 1 || rank < 0 || rank >= n_ranks) return fail(B200_ERR_INVALID_ARGUMENT, "bad communicator arguments");
    *out = nullptr;
    if (!nccl().ok) return fail(B200_ERR_UNSUPPORTED, "libnccl.so.2 could not be loaded");
    if (device < 0 && cudaGetDevice(&device) != cudaSuccess) return cuda_fail(nullptr, cudaGetLastError(), "cudaGetDevice");
    if (cudaSetDevice(device) != cudaSuccess) return cuda_fail(nullptr, cudaGetLastError(), "cudaSetDevice");
    ncclUniqueId id;
    std::memcpy(&id, id_bytes, sizeof id);
    b200_comm *c = new (std::nothrow) b200_comm();
    if (!c) return fail(B200_ERR_OUT_OF_MEMORY, "out of host memory");
    c->n_ranks = n_ranks; c->rank = rank; c->device = device;
    ncclResult_t r = nccl().CommInitRank(&c->comm, n_ranks, id, rank);
    if (r != ncclSuccess) { delete c; return nccl_fail(r, "ncclCommInitRank"); }
    cudaEventCreate(&c->ev0);
    cudaEventCreate(&c->ev1);
    *out = c;
    return B200_OK;
}

void b200_comm_destroy(b200_comm *c)
{
    if (!c) return;
    cudaSetDevice(c->device);
    b200_comm_peer_detach(c);
    if (c->send) cudaFree(c->send);
    if (c->recv) cudaFree(c->recv);
    if (c->ev0) cudaEventDestroy(c->ev0);
    if (c->ev1) cudaEventDestroy(c->ev1);
    if (c->comm && nccl().ok) nccl().CommDestroy(c->comm);
    (void)cudaGetLastError();
    delete c;
}

int b200_comm_rank(const b200_comm *c) { return c ? c->rank : -1; }
int b200_comm_size(const b200_comm *c) { return c ? c->n_ranks : 0; }
double b200_comm_last_ms(const b200_comm *c) { return c ? c->last_ms : 0.0; }

uint64_t b200_sixdof_trajectory_gather_bytes(const b200_sixdof *h, const uint64_t *worlds_per_rank, int n_ranks)
{
    if (!h || !worlds_per_rank) return 0;
    uint64_t worlds = 0;
    for (int r = 0; r < n_ranks; ++r) worlds += worlds_per_rank[r];
    return worlds * b200_sixdof_trajectory_len(h) * h->desc.n_entities * (uint64_t)h->traj_planes * 8ull;
}

// World-sharded all-gather of the trajectory ring: rank r holds worlds_per_rank[r] worlds (every rank the same
// number of samples, entities and ring width); afterwards `dst` on every rank holds
// [sum(worlds)][samples][n_entities][width] in rank order.  dst may be a device or a host pointer.
int b200_sixdof_trajectory_allgather(b200_sixdof *h, b200_comm *c, const uint64_t *worlds_per_rank, void *dst, uint64_t dst_bytes)
{
    if (!h || !c || !worlds_per_rank || !dst) return fail(B200_ERR_INVALID_ARGUMENT, "null argument");
    if (h->status != B200_OK) return fail(h->status, "handle is in a failed state");
    if (h->device != c->device) return fail(B200_ERR_INVALID_ARGUMENT, "handle is on device %d, communicator on %d", h->device, c->device);
    CU(h, cudaSetDevice(h->device));
    if (worlds_per_rank[c->rank] != h->desc.n_worlds)
        return fail(B200_ERR_VALUE_SIZE_MISMATCH, "rank %d holds %llu worlds, worlds_per_rank says %llu", c->rank,
                    (unsigned long long)h->desc.n_worlds, (unsigned long long)worlds_per_rank[c->rank]);
    const uint64_t S = b200_sixdof_trajectory_len(h), N = h->desc.n_entities, W = h->traj_planes;
    const uint64_t want = b200_sixdof_trajectory_gather_bytes(h, worlds_per_rank, c->n_ranks);
    if (dst_bytes != want) return fail(B200_ERR_VALUE_SIZE_MISMATCH, "gathered trajectory is %llu bytes, got %llu", (unsigned long long)want, (unsigned long long)dst_bytes);
    if (want == 0) return B200_OK;
    const uint64_t row = S * N * W; // doubles per world
    const uint64_t mine = h->desc.n_worlds * row;
    if (c->send_bytes < mine * 8) {
        if (c->send) CU(h, cudaFree(c->send));
        c->send = nullptr; c->send_bytes = 0;
        CU(h, cudaMalloc(&c->send, std::max<uint64_t>(mine * 8, 8)));
        c->send_bytes = mine * 8;
    }
    cudaPointerAttributes at{};
    const bool dst_dev = cudaPointerGetAttributes(&at, dst) == cudaSuccess && at.type == cudaMemoryTypeDevice;
    (void)cudaGetLastError();
    double *recv = (double *)dst;
    if (!dst_dev) {
        if (c->recv_bytes < want) {
            if (c->recv) CU(h, cudaFree(c->recv));
            c->recv = nullptr; c->recv_bytes = 0;
            CU(h, cudaMalloc(&c->recv, want));
            c->recv_bytes = want;
        }
        recv = c->recv;
    }
    CU(h, cudaEventRecord(c->ev0, h->stream));
    if (mine) {
        const size_t smem = (size_t)kGTile * (W | 1u) * sizeof(double);
        for (uint64_t s0 = 0; s0 < S; s0 += 32768) {
            const dim3 grid((unsigned)((h->n_bodies + kGTile - 1) / kGTile), (unsigned)std::min<uint64_t>(32768, S - s0));
            // the kernel indexes samples from blockIdx.y: shift the ring, and the output by s0 rows of N*W inside each world
            traj_world_major_kernel<<<grid, kGTile, smem, h->stream>>>(h->traj + s0 * W * h->ld, c->send + s0 * N * W, h->n_bodies,
                                                                     (uint32_t)N, (uint32_t)W, S, h->ld);
        }
        CU(h, cudaGetLastError());
        h->timings.kernel_launches++;
    }
    bool even = true;
    for (int r = 0; r < c->n_ranks; ++r) even = even && worlds_per_rank[r] == worlds_per_rank[0];
    if (even) {
        NC(nccl().AllGather(c->send, recv, mine, ncclDouble, c->comm, h->stream));
    } else {
        // ragged shards: one broadcast per rank, fused into one NCCL group
        NC(nccl().GroupStart());
        uint64_t off = 0;
        for (int r = 0; r < c->n_ranks; ++r) {
            const uint64_t cnt = worlds_per_rank[r] * row;
            if (cnt) {
                ncclResult_t rr = nccl().Broadcast(c->send, recv + off, cnt, ncclDouble, r, c->comm, h->stream);
                if (rr != ncclSuccess) { nccl().GroupEnd(); return nccl_fail(rr, "ncclBroadcast"); }
            }
            off += cnt;
        }
        NC(nccl().GroupEnd());
    }
    CU(h, cudaEventRecord(c->ev1, h->stream));
    if (!dst_dev) CU(h, cudaMemcpyAsync(dst, recv, want, cudaMemcpyDeviceToHost, h->stream));
    CU(h, cudaStreamSynchronize(h->stream));
    float ms = 0.f;
    cudaEventElapsedTime(&ms, c->ev0, c->ev1);
    c->last_ms = ms; // layout kernel + collective, device-timed on the handle's stream
    return B200_OK;
}

// Peer window for the row-sharded world: every rank allocates X[2][6][ld] + delivery counters, the ranks swap the CUDA
// IPC handles of those allocations through the communicator, and each maps all the others.  From then on
// b200_sixdof_step_row_sharded exchanges the rows with direct NVLink stores and counter releases — no collective in
// the tick loop.  Collective call: every rank of the communicator must make it, with handles of the same shape.
int b200_comm_peer_attach(b200_comm *c, b200_sixdof *h)
{
    if (!h || !c) return fail(B200_ERR_INVALID_ARGUMENT, "null argument");
    if (h->device != c->device) return fail(B200_ERR_INVALID_ARGUMENT, "handle is on device %d, communicator on %d", h->device, c->device);
    if (c->n_ranks > B200_MAX_PEERS) return fail(B200_ERR_UNSUPPORTED, "peer windows support up to %d ranks", B200_MAX_PEERS);
    CU(h, cudaSetDevice(h->device));
    b200_comm_peer_detach(c);
    auto &w = c->win;
    w.ld = h->ld;
    char *mem = nullptr;
    CU(h, cudaMalloc(&mem, win_bytes(w.ld) + 64));
    CU(h, cudaMemsetAsync(mem, 0, win_bytes(w.ld) + 64, h->stream));
    w.base[c->rank] = (double *)mem;
    w.ctr = (unsigned *)(mem + win_bytes(w.ld));
    // swap the IPC handles (64 bytes each) over the communicator
    cudaIpcMemHandle_t mine{}, all[B200_MAX_PEERS];
    cudaError_t e = cudaIpcGetMemHandle(&mine, mem);
    char *xs = nullptr;
    int rc = B200_OK;
    if (e != cudaSuccess) { (void)cudaGetLastError(); rc = fail(B200_ERR_UNSUPPORTED, "CUDA IPC export failed: %s", cudaGetErrorString(e)); }
    if (cudaMalloc(&xs, sizeof(mine) * (size_t)(c->n_ranks + 1)) != cudaSuccess) { // nothing collective has started yet
        (void)cudaGetLastError();
        cudaFree(mem);
        w.base[c->rank] = nullptr;
        return fail(B200_ERR_OUT_OF_MEMORY, "out of device memory");
    }
    if (!rc && cudaMemcpyAsync(xs, &mine, sizeof mine, cudaMemcpyHostToDevice, h->stream) != cudaSuccess) rc = cuda_fail(h, cudaGetLastError(), "cudaMemcpyAsync(ipc handle)");
    {   // every rank takes part in the exchange even after a local failure (its handle is then all zeros)
        ncclResult_t r = nccl().AllGather(xs, xs + sizeof mine, sizeof mine, ncclChar, c->comm, h->stream);
        if (r != ncclSuccess && !rc) rc = nccl_fail(r, "ncclAllGather(ipc handles)");
    }
    if (!rc && (cudaMemcpyAsync(all, xs + sizeof mine, sizeof(mine) * (size_t)c->n_ranks, cudaMemcpyDeviceToHost, h->stream) != cudaSuccess ||
                cudaStreamSynchronize(h->stream) != cudaSuccess))
        rc = cuda_fail(h, cudaGetLastError(), "ipc handle exchange");
    cudaFree(xs);
    for (int r = 0; r < c->n_ranks && !rc; ++r) {
        if (r == c->rank) continue;
        void *p = nullptr;
        e = cudaIpcOpenMemHandle(&p, all[r], cudaIpcMemLazyEnablePeerAccess);
        if (e != cudaSuccess) { (void)cudaGetLastError(); rc = fail(B200_ERR_UNSUPPORTED, "CUDA IPC import of rank %d's window failed: %s", r, cudaGetErrorString(e)); }
        else w.base[r] = (double *)p;
    }
    // every rank learns whether every rank mapped every window: all attach or none does
    int ok_all = 0;
    {
        int *flags = nullptr;
        if (cudaMalloc(&flags, sizeof(int) * (size_t)(c->n_ranks + 1)) == cudaSuccess) {
            int mine_ok = rc == B200_OK ? 1 : 0, got[B200_MAX_PEERS] = {};
            cudaMemcpyAsync(flags, &mine_ok, sizeof(int), cudaMemcpyHostToDevice, h->stream);
            if (nccl().AllGather(flags, flags + 1, 1, ncclInt32, c->comm, h->stream) == ncclSuccess &&
                cudaMemcpyAsync(got, flags + 1, sizeof(int) * (size_t)c->n_ranks, cudaMemcpyDeviceToHost, h->stream) == cudaSuccess &&
                cudaStreamSynchronize(h->stream) == cudaSuccess) {
                ok_all = 1;
                for (int r = 0; r < c->n_ranks; ++r) ok_all &= got[r];
            }
            cudaFree(flags);
        }
        (void)cudaGetLastError();
    }
    if (!ok_all) {
        b200_comm_peer_detach(c);
        return rc ? rc : fail(B200_ERR_UNSUPPORTED, "another rank could not map the peer windows");
    }
    w.owner = h;
    w.owner_serial = h->serial;
    return B200_OK;
}

int b200_comm_peer_attached(const b200_comm *c) { return c && c->win.owner ? 1 : 0; }

// Collective when a window exists: every rank unmaps its imports, then (after a tiny all-gather as the barrier) frees
// its own allocation — freeing memory a peer still maps is undefined.
void b200_comm_peer_detach(b200_comm *c)
{
    if (!c || !c->win.base[c->rank]) return;
    cudaSetDevice(c->device);
    cudaDeviceSynchronize();
    for (int r = 0; r < B200_MAX_PEERS; ++r) {
        if (!c->win.base[r] || r == c->rank) continue;
        cudaIpcCloseMemHandle(c->win.base[r]);
        c->win.base[r] = nullptr;
    }
    if (c->comm && nccl().ok && c->n_ranks > 1) {
        int *b = nullptr;
        if (cudaMalloc(&b, sizeof(int) * (size_t)(c->n_ranks + 1)) == cudaSuccess) {
            cudaMemset(b, 0, sizeof(int) * (size_t)(c->n_ranks + 1));
            if (nccl().AllGather(b, b + 1, 1, ncclInt32, c->comm, nullptr) == ncclSuccess) cudaDeviceSynchronize();
            cudaFree(b);
        }
    }
    cudaFree(c->win.base[c->rank]);
    c->win.base[c->rank] = nullptr;
    c->win.ctr = nullptr;
    c->win.owner = nullptr;
    (void)cudaGetLastError();
}

// One world, rows split over the ranks of `c` (SURVEY §8e, second case).  Every rank holds the whole world (same
// handle description, same initial state) but folds and integrates only its own source rows
// [rank * N / R, (rank + 1) * N / R); after each tick the rows' new linear position and velocity planes — all the
// other ranks' gravity needs — are exchanged with an in-place ncclAllGather per plane (one NCCL group per tick,
// 6 planes x N/R doubles per rank over NVLink); the last tick of the call gathers every plane of WorldPos, WorldVel,
// WorldAccel and Force so that each rank ends with the complete world.  Stage positions depend on the tick's input
// state only (rk4.rs:85-111), so one exchange per tick suffices.
int b200_sixdof_step_row_sharded(b200_sixdof *h, b200_comm *c, uint64_t n_ticks)
{
    if (!h || !c) return fail(B200_ERR_INVALID_ARGUMENT, "null argument");
    if (h->status != B200_OK) return fail(h->status, "handle is in a failed state");
    if (!h->schedules.empty())
        return fail(B200_ERR_UNSUPPORTED, "b200_sixdof_step_row_sharded does not support input schedules (clear them first)");
    if (h->device != c->device) return fail(B200_ERR_INVALID_ARGUMENT, "handle is on device %d, communicator on %d", h->device, c->device);
    if (h->graph_eff < 0 || !h->graph_dense || h->desc.n_worlds != 1 || h->egm_eff >= 0)
        return fail(B200_ERR_UNSUPPORTED, "row sharding applies to one world with dense (all-pairs) edge_fold gravity (and no EGM08 effector)");
    const uint64_t N = h->desc.n_entities, R = (uint64_t)c->n_ranks;
    if (N % R != 0) return fail(B200_ERR_UNSUPPORTED, "row sharding needs n_entities (%llu) divisible by the rank count (%llu)", (unsigned long long)N, (unsigned long long)R);
    CU(h, cudaSetDevice(h->device));
    const uint64_t rows = N / R, i0 = rows * (uint64_t)c->rank;
    const bool exact = h->desc.math_mode == B200_MATH_EXACT;
    const b200_effector &e = h->effectors[h->graph_eff];
    static const int peer_env = env_int("B200_ROW_PEER", 1);
    // (a window attached to another handle — or to a destroyed one whose address this handle reuses — is ignored)
    const bool peer = peer_env && c->win.owner == h && c->win.owner_serial == h->serial && c->win.ld == h->ld;
    double *const pos = h->find(B200_ID_WORLD_POS)->dev, *const vel = h->find(B200_ID_WORLD_VEL)->dev;
    double *const acc = h->find(B200_ID_WORLD_ACCEL)->dev, *const frc = h->find(B200_ID_FORCE)->dev;
    auto gather_plane = [&](double *plane) { return nccl().AllGather(plane + i0, plane, rows, ncclDouble, c->comm, h->stream); };
    unsigned long long *const flags = peer ? (unsigned long long *)(c->win.base[c->rank] + win_doubles(h->ld)) : nullptr;
    if (peer) {
        // the window's current-parity half <- the local world (covers uploads and non-sharded steps since the last call)
        const unsigned long long T = h->ticks_done;
        peer_fill_kernel<<<(unsigned)((N + 255) / 256), 256, 0, h->stream>>>(pos, vel, c->win.base[c->rank] + (T & 1ull) * 6ull * h->ld, flags,
                                                                             h->ld, (uint32_t)N, (int)R, T);
        CU(h, cudaGetLastError());
        h->timings.kernel_launches++;
    }
    for (uint64_t t = 0; t < n_ticks; ++t) {
        const bool last = t + 1 == n_ticks;
        const unsigned long long T = h->ticks_done + t;
        StepParams P;
        fill_step_params(h, P);
        GraphParams G{};
        G.pos = P.pos; G.vel = P.vel; G.ine = P.ine; G.gforce = h->gforce;
        G.ld = h->ld; G.n_entities = (uint32_t)N; G.n_worlds = 1;
        G.dt_stage = P.dt_stage; G.kind = e.kind; G.integrator = h->desc.integrator;
        G.p0 = e.p[0]; G.p1 = e.p[1]; G.row_ptr = h->row_ptr; G.col_idx = h->col_idx; G.max_deg = h->max_deg;
        G.src0 = (uint32_t)i0; G.src_n = (uint32_t)rows;
        if (peer) {
            // gravity reads every row's x, v from the window half of this tick count (the fold kernels touch planes
            // 4..6 of pos and 3..5 of vel only), once every rank's rows of that count have landed
            const double *X = c->win.base[c->rank] + (T & 1ull) * 6ull * h->ld;
            G.pos = X - 4 * h->ld;
            G.vel = X;
            if (t == 0) { // later ticks: the previous tick's push kernel already waited
                peer_wait_kernel<<<1, 32, 0, h->stream>>>(flags, (int)R, T);
                h->timings.kernel_launches++;
            }
        }
        CU(h, launch_graph_force(G, (int)h->desc.math_mode, true, h->stream));
        // the body kernel on this rank's rows only: shift every per-body plane, keep the entity numbering
        P.pos += i0; P.vel += i0; P.acc += i0; P.frc += i0; P.ine += i0;
        if (P.gforce) P.gforce += i0;
        if (P.traj) P.traj += i0;
        for (uint32_t k = 0; k < P.n_eff; ++k) if (P.eff[k].col) P.eff[k].col += i0;
        P.n_bodies = rows;
        P.ent0 = (uint32_t)i0;
        P.n_ticks = 1;
        P.tick0 = T;
        P.write_fa = (exact || last) ? 1u : 0u;
        CU(h, launch_body_step(P, (int)h->desc.integrator, (int)h->desc.math_mode, h->stream));
        h->timings.kernel_launches += 2;
        if (peer) {
            // exchange: this rank's new x, v rows straight into every rank's next-parity half, then one counter release each
            PeerPush a{};
            a.pos = pos + i0; a.vel = vel + i0; a.ctr = c->win.ctr;
            a.wait = last ? nullptr : flags;
            a.ld_src = a.ld_dst = h->ld; a.rows = (uint32_t)rows; a.n_ranks = (int)R; a.value = T + 1;
            for (uint64_t r = 0; r < R; ++r) {
                a.dst[r] = c->win.base[r] + ((T + 1) & 1ull) * 6ull * h->ld + i0;
                a.flag[r] = (unsigned long long *)(c->win.base[r] + win_doubles(h->ld)) + c->rank;
            }
            peer_push_kernel<<<dim3((unsigned)((rows + 127) / 128), 6), 128, 0, h->stream>>>(a);
            CU(h, cudaGetLastError());
            h->timings.kernel_launches++;
            if (!last) continue;
        }
        // exchange over NCCL: in-place all-gather of the row slices, plane by plane (every tick without a peer window;
        // with one, only the call's last tick, which completes the attitude / accel / force planes of the other ranks' rows)
        NC(nccl().GroupStart());
        ncclResult_t r = ncclSuccess;
        for (int k = 0; k < 7 && r == ncclSuccess; ++k) if (last || k >= 4) r = gather_plane(pos + (uint64_t)k * h->ld);
        for (int k = 0; k < 6 && r == ncclSuccess; ++k) if (last || k >= 3) r = gather_plane(vel + (uint64_t)k * h->ld);
        if (last) {
            for (int k = 0; k < 6 && r == ncclSuccess; ++k) r = gather_plane(acc + (uint64_t)k * h->ld);
            for (int k = 0; k < 6 && r == ncclSuccess; ++k) r = gather_plane(frc + (uint64_t)k * h->ld);
        }
        if (r != ncclSuccess) { nccl().GroupEnd(); return nccl_fail(r, "ncclAllGather(row slice)"); }
        NC(nccl().GroupEnd());
    }
    h->ticks_done += n_ticks;
    h->tick += n_ticks;
    h->timings.ticks += n_ticks;
    return B200_OK;
}

// Concurrent host<->device bandwidth of one GPU (pinned `host` of >= max(h2d, d2h) * 2 bytes): an H2D stream and a
// D2H stream run `iters` copies each at the same time; out[0] = H2D GB/s, out[1] = D2H GB/s.  bench.py runs it on
// every rank at once to report the PCIe / host-memory ceiling its e2e number sits under.
// The same measurement with kernels instead of the copy engines: SMs read mapped pinned host memory (H2D leg) and write it
// (D2H leg), both at once on two streams, `blocks` CTAs of 256 threads per leg.  out[0] = H2D GB/s, out[1] = D2H GB/s.
int b200_probe_zero_copy_gbs(int device, void *host, uint64_t h2d_bytes, uint64_t d2h_bytes, int iters, int blocks, double *out)
{
    if (!host || !out || iters < 1 || blocks < 1) return fail(B200_ERR_INVALID_ARGUMENT, "bad arguments");
    if (b200_device_count() <= 0) return B200_ERR_NO_DEVICE;
    if (device >= 0 && cudaSetDevice(device) != cudaSuccess) return cuda_fail(nullptr, cudaGetLastError(), "cudaSetDevice");
    void *hdev = nullptr;
    if (cudaHostGetDevicePointer(&hdev, host, 0) != cudaSuccess) { (void)cudaGetLastError(); return fail(B200_ERR_UNSUPPORTED, "host buffer is not mapped into the device address space"); }
    void *din = nullptr, *dout = nullptr;
    cudaStream_t s0 = nullptr, s1 = nullptr;
    cudaEvent_t e[4] = {nullptr, nullptr, nullptr, nullptr};
    int rc = B200_OK;
    if (cudaMalloc(&din, std::max<uint64_t>(h2d_bytes, 16)) != cudaSuccess || cudaMalloc(&dout, std::max<uint64_t>(d2h_bytes, 16)) != cudaSuccess)
        rc = cuda_fail(nullptr, cudaGetLastError(), "cudaMalloc(probe)");
    if (!rc) {
        cudaStreamCreateWithFlags(&s0, cudaStreamNonBlocking);
        cudaStreamCreateWithFlags(&s1, cudaStreamNonBlocking);
        for (auto &x : e) cudaEventCreate(&x);
        char *hin = (char *)hdev, *hout = (char *)hdev + h2d_bytes;
        for (int w = 0; w < 2; ++w) {
            cudaEventRecord(e[0], s0); cudaEventRecord(e[2], s1);
            for (int i = 0; i < (w ? iters : 1); ++i) {
                if (h2d_bytes) copy16_kernel<<<blocks, 256, 0, s0>>>((const double2 *)hin, (double2 *)din, h2d_bytes / 16);
                if (d2h_bytes) copy16_kernel<<<blocks, 256, 0, s1>>>((const double2 *)dout, (double2 *)hout, d2h_bytes / 16);
            }
            cudaEventRecord(e[1], s0); cudaEventRecord(e[3], s1);
            cudaStreamSynchronize(s0); cudaStreamSynchronize(s1);
        }
        float m0 = 0.f, m1 = 0.f;
        cudaEventElapsedTime(&m0, e[0], e[1]);
        cudaEventElapsedTime(&m1, e[2], e[3]);
        out[0] = m0 > 0 ? (double)h2d_bytes * iters / (m0 * 1e-3) / 1e9 : 0.0;
        out[1] = m1 > 0 ? (double)d2h_bytes * iters / (m1 * 1e-3) / 1e9 : 0.0;
        if (cudaGetLastError() != cudaSuccess) rc = fail(B200_ERR_CUDA, "zero-copy probe failed");
    }
    for (auto &x : e) if (x) cudaEventDestroy(x);
    if (s0) cudaStreamDestroy(s0);
    if (s1) cudaStreamDestroy(s1);
    if (din) cudaFree(din);
    if (dout) cudaFree(dout);
    return rc;
}

int b200_probe_pcie_gbs(int device, void *host, uint64_t h2d_bytes, uint64_t d2h_bytes, int iters, double *out)
{
    if (!host || !out || iters < 1) return fail(B200_ERR_INVALID_ARGUMENT, "bad arguments");
    if (b200_device_count() <= 0) return B200_ERR_NO_DEVICE;
    if (device >= 0 && cudaSetDevice(device) != cudaSuccess) return cuda_fail(nullptr, cudaGetLastError(), "cudaSetDevice");
    void *din = nullptr, *dout = nullptr;
    cudaStream_t s0 = nullptr, s1 = nullptr;
    cudaEvent_t e[4] = {nullptr, nullptr, nullptr, nullptr};
    int rc = B200_OK;
    if (cudaMalloc(&din, std::max<uint64_t>(h2d_bytes, 8)) != cudaSuccess || cudaMalloc(&dout, std::max<uint64_t>(d2h_bytes, 8)) != cudaSuccess)
        rc = cuda_fail(nullptr, cudaGetLastError(), "cudaMalloc(probe)");
    if (!rc) {
        cudaStreamCreateWithFlags(&s0, cudaStreamNonBlocking);
        cudaStreamCreateWithFlags(&s1, cudaStreamNonBlocking);
        for (auto &x : e) cudaEventCreate(&x);
        char *hin = (char *)host, *hout = (char *)host + h2d_bytes;
        for (int w = 0; w < 2; ++w) { // warm-up pass, then the timed pass
            cudaEventRecord(e[0], s0); cudaEventRecord(e[2], s1);
            for (int i = 0; i < (w ? iters : 1); ++i) {
                if (h2d_bytes) cudaMemcpyAsync(din, hin, h2d_bytes, cudaMemcpyHostToDevice, s0);
                if (d2h_bytes) cudaMemcpyAsync(hout, dout, d2h_bytes, cudaMemcpyDeviceToHost, s1);
            }
            cudaEventRecord(e[1], s0); cudaEventRecord(e[3], s1);
            cudaStreamSynchronize(s0); cudaStreamSynchronize(s1);
        }
        float m0 = 0.f, m1 = 0.f;
        cudaEventElapsedTime(&m0, e[0], e[1]);
        cudaEventElapsedTime(&m1, e[2], e[3]);
        out[0] = m0 > 0 ? (double)h2d_bytes * iters / (m0 * 1e-3) / 1e9 : 0.0;
        out[1] = m1 > 0 ? (double)d2h_bytes * iters / (m1 * 1e-3) / 1e9 : 0.0;
        if (cudaGetLastError() != cudaSuccess) rc = fail(B200_ERR_CUDA, "PCIe probe failed");
    }
    for (auto &x : e) if (x) cudaEventDestroy(x);
    if (s0) cudaStreamDestroy(s0);
    if (s1) cudaStreamDestroy(s1);
    if (din) cudaFree(din);
    if (dout) cudaFree(dout);
    return rc;
}

} // extern "C"
