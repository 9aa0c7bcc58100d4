// psx.cu -- host runtime + C ABI (include/psx.h) of the B200 parameter-server
// data plane.  One process per GPU is the normal deployment (the process that
// replaces tf.train.Server at tfmesos/server.py:51-66); several devices in one
// process also work (every object remembers its device).
//
// Memory model
//   shard   = ONE cudaMalloc on the PS GPU:  [header 4 KiB | var | m | v | slots]
//             exported with CUDA IPC; workers map the whole thing and write
//             their gradient slot + its flag word directly over NVLink.
//   client  = a worker's attachment to a shard: mapped pointers + a 256 B block
//             in the WORKER's HBM (push ticket, mirror of apply_seq).
//   buffer  = exportable worker staging (gradients / parameters) for psx_round.
// Waiting never holds an SM: consumers wait with cuStreamWaitValue32 on a flag
// in their OWN HBM that the producer's kernel publishes remotely (fence.sys + store).
#include <cuda.h>
#include <cuda_runtime.h>
#include <unistd.h>

#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <thread>
#include <unordered_map>
#include <vector>

#include "psx.h"
#include "psx_kernels.cuh"

using namespace psx;

namespace {

// ------------------------------------------------------------------ errors --
thread_local char g_err[512] = "";

int fail(int code, const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

#define CU_TRY(expr)                                                                   \
    do {                                                                               \
        cudaError_t e_ = (expr);                                                       \
        if (e_ != cudaSuccess)                                                         \
            return fail(PSX_ECUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e_), \
                        __FILE__, __LINE__);                                           \
    } while (0)

// Entry points run on the object's device and put the caller's device back
// (torch tracks the thread's current device through the same driver state).
struct DeviceGuard {
    int prev = -1;
    cudaError_t err = cudaSuccess;
    explicit DeviceGuard(int device)
    {
        err = cudaGetDevice(&prev);
        if (err == cudaSuccess && prev != device) err = cudaSetDevice(device);
        else if (err == cudaSuccess) prev = -1;
    }
    ~DeviceGuard()
    {
        if (prev >= 0) cudaSetDevice(prev);
    }
};
#define PSX_DEVICE(dev)                                                                  \
    DeviceGuard guard_(dev);                                                             \
    if (guard_.err != cudaSuccess)                                                       \
        return fail(PSX_ECUDA, "selecting device %d: %s", (int)(dev), cudaGetErrorString(guard_.err))

// ------------------------------------------------------------ driver memops --
typedef CUresult (*WaitValue32Fn)(CUstream, CUdeviceptr, cuuint32_t, unsigned int);
WaitValue32Fn g_wait32 = nullptr;
std::once_flag g_wait_once;

int resolve_memops()
{
    std::call_once(g_wait_once, [] {
        void *fn = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuStreamWaitValue32", &fn, cudaEnableDefault, &q) ==
                cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            g_wait32 = (WaitValue32Fn)fn;
    });
    if (!g_wait32) return fail(PSX_ECUDA, "cuStreamWaitValue32 not available from the driver");
    return PSX_OK;
}

int stream_wait_geq(void *stream, unsigned int *flag, uint32_t value)
{
    int rc = resolve_memops();
    if (rc) return rc;
    CUresult r = g_wait32((CUstream)stream, (CUdeviceptr)(uintptr_t)flag, value,
                          CU_STREAM_WAIT_VALUE_GEQ);
    if (r != CUDA_SUCCESS) return fail(PSX_ECUDA, "cuStreamWaitValue32 failed: CUresult %d", (int)r);
    return PSX_OK;
}

// ---------------------------------------------------------------- objects ---
constexpr uint32_t kMagic = 0x50535831u;  // "PSX1"
constexpr size_t kHeaderBytes = 4096;
constexpr uint64_t kPadElems = 1024;      // every region starts 4 KiB aligned

enum Kind : uint32_t { KIND_SHARD = 1, KIND_CLIENT = 2, KIND_BUFFER = 3, KIND_MAILBOX = 4 };

struct HandleBlob {           // PSX_HANDLE_BYTES, shipped between processes
    uint32_t magic, abi, kind;
    int32_t device;
    uint64_t pid, local_id, nelem, nelem_pad;
    int32_t opt, n_slots, wire;
    uint32_t pad;
    cudaIpcMemHandle_t ipc;
};
static_assert(sizeof(HandleBlob) == PSX_HANDLE_BYTES, "handle blob size");

// f32 state arrays the optimizer keeps beside var (OptTraits::kState); -1: unknown id
int state_arrays(int opt)
{
    switch (opt) {
    case PSX_OPT_SGD: return OptTraits<PSX_OPT_SGD>::kState;
    case PSX_OPT_ADAM: return OptTraits<PSX_OPT_ADAM>::kState;
    case PSX_OPT_MOMENTUM: return OptTraits<PSX_OPT_MOMENTUM>::kState;
    case PSX_OPT_ADAGRAD: return OptTraits<PSX_OPT_ADAGRAD>::kState;
    case PSX_OPT_RMSPROP: return OptTraits<PSX_OPT_RMSPROP>::kState;
    default: return -1;
    }
}

struct Layout {
    uint64_t nelem = 0, nelem_pad = 0;
    int opt = 0, n_slots = 0, wire = 0;
    size_t wire_bytes() const { return wire == PSX_BF16 ? 2 : 4; }
    int n_state() const { return state_arrays(opt); }
    size_t off_var() const { return kHeaderBytes; }
    size_t off_m() const { return off_var() + nelem_pad * 4; }
    size_t off_v() const { return off_m() + (n_state() >= 1 ? nelem_pad * 4 : 0); }
    size_t off_slots() const { return off_v() + (n_state() >= 2 ? nelem_pad * 4 : 0); }
    size_t total() const { return off_slots() + (size_t)n_slots * nelem_pad * wire_bytes(); }
};

struct Mapped {               // a peer allocation opened in this process
    char *base = nullptr;
    bool ipc = false;         // needs cudaIpcCloseMemHandle
    int device = 0;
};

struct Bound {
    Mapped grad, param;
    uint64_t elem_off = 0;
    bool valid = false;
};

struct Server;
struct Shard {
    int device = 0;
    Server *server = nullptr;         // request-free serving loop (psx_serve_start)
    std::recursive_mutex serve_mu;    // start / stop / pause of that loop: accessors may come
                                      // from several endpoint threads at once
    Layout lay;
    char *base = nullptr;
    int sm_count = 148;
    Mapped client_map[PSX_MAX_SLOTS];
    unsigned int *mirror[PSX_MAX_SLOTS] = {};
    Bound bound[PSX_MAX_SLOTS];
    Mapped mailbox_map[PSX_MAX_SLOTS];
    unsigned int *mailbox[PSX_MAX_SLOTS] = {};
    const float *mc_grad = nullptr;   // NVLS binding (psx_round_bind_mc): multicast addresses
    float *mc_param = nullptr;        // of this shard's range in the workers' arena
    int mc_members = 0;
    ShardHeader *hdr() const { return (ShardHeader *)base; }
    float *var() const { return (float *)(base + lay.off_var()); }
    float *m() const { return (float *)(base + lay.off_m()); }
    float *v() const { return (float *)(base + lay.off_v()); }
    char *slot(int s) const { return base + lay.off_slots() + (size_t)s * lay.nelem_pad * lay.wire_bytes(); }
};

struct Client {
    int device = 0;           // the worker's device
    int slot = 0;
    Layout lay;
    Mapped shard;             // the PS allocation as seen from here
    ClientBlock *block = nullptr;  // in this device's HBM
    cudaStream_t poll_stream = nullptr;   // psx_client_poll's private stream
    int sm_count = 148;
    ShardHeader *hdr() const { return (ShardHeader *)shard.base; }
    float *var() const { return (float *)(shard.base + lay.off_var()); }
    char *my_slot() const { return shard.base + lay.off_slots() + (size_t)slot * lay.nelem_pad * lay.wire_bytes(); }
};

struct Mailbox {              // a worker's completion counter, in ITS HBM
    int device = 0;
    unsigned int *counter = nullptr;
};

struct TensorList {
    uint64_t client_id = 0;
    int device = 0;
    ListChunk *d_chunks = nullptr;
    int n_chunks = 0;
    int sm_count = 148;
};

struct Buffer {
    int device = 0;
    uint64_t nbytes = 0;
    char *base = nullptr;
};

std::mutex g_mu;
std::unordered_map<uint64_t, Shard *> g_shards;
std::unordered_map<uint64_t, Client *> g_clients;
std::unordered_map<uint64_t, Buffer *> g_buffers;
std::unordered_map<uint64_t, TensorList *> g_lists;
std::unordered_map<uint64_t, Mailbox *> g_mailboxes;
std::atomic<uint64_t> g_next_id{1};
std::atomic<uint64_t> g_launches{0};

template <typename T> T *find(std::unordered_map<uint64_t, T *> &m, uint64_t id)
{
    std::lock_guard<std::mutex> lk(g_mu);
    auto it = m.find(id);
    return it == m.end() ? nullptr : it->second;
}

int sm_count_of(int device)
{
    int n = 148;
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, device);
    return n > 0 ? n : 148;
}

int enable_peer(int device, int peer);

// Maps the object a handle names for use from `device`.  Same process: the raw
// pointer, after enabling peer access between the two ordinals.  Other process:
// CUDA IPC, which enables peer access itself (the exporter's ordinal means
// nothing here -- the importer may see a different set of GPUs through
// CUDA_VISIBLE_DEVICES, as tfrun -Gw 1 workers do).
int open_blob(const HandleBlob &b, int device, Mapped *out)
{
    out->device = b.device;
    if (b.pid == (uint64_t)getpid()) {  // same process: direct pointer
        int prc = enable_peer(device, b.device);
        if (prc) return prc;
        std::lock_guard<std::mutex> lk(g_mu);
        char *base = nullptr;
        if (b.kind == KIND_SHARD) {
            auto it = g_shards.find(b.local_id);
            if (it != g_shards.end()) base = it->second->base;
        } else if (b.kind == KIND_CLIENT) {
            auto it = g_clients.find(b.local_id);
            if (it != g_clients.end()) base = (char *)it->second->block;
        } else if (b.kind == KIND_BUFFER) {
            auto it = g_buffers.find(b.local_id);
            if (it != g_buffers.end()) base = it->second->base;
        } else if (b.kind == KIND_MAILBOX) {
            auto it = g_mailboxes.find(b.local_id);
            if (it != g_mailboxes.end()) base = (char *)it->second->counter;
        }
        if (!base) return fail(PSX_EINVAL, "handle refers to an object this process no longer has");
        out->base = base;
        out->ipc = false;
        return PSX_OK;
    }
    PSX_DEVICE(device);
    void *p = nullptr;
    CU_TRY(cudaIpcOpenMemHandle(&p, b.ipc, cudaIpcMemLazyEnablePeerAccess));
    out->base = (char *)p;
    out->ipc = true;
    return PSX_OK;
}

void close_mapped(Mapped &m)
{
    if (m.ipc && m.base) cudaIpcCloseMemHandle(m.base);
    m.base = nullptr;
    m.ipc = false;
}

int check_blob(const void *handle, uint32_t kind, HandleBlob *out)
{
    if (!handle) return fail(PSX_EINVAL, "null handle");
    memcpy(out, handle, sizeof(HandleBlob));
    if (out->magic != kMagic) return fail(PSX_EINVAL, "not a psx handle");
    if (out->abi != PSX_ABI_VERSION)
        return fail(PSX_EABI, "handle from ABI %u, library is ABI %d", out->abi, PSX_ABI_VERSION);
    if (out->kind != kind) return fail(PSX_EINVAL, "handle kind %u, expected %u", out->kind, kind);
    return PSX_OK;
}

int enable_peer(int device, int peer)
{
    if (device == peer) return PSX_OK;
    int can = 0;
    CU_TRY(cudaDeviceCanAccessPeer(&can, device, peer));
    if (!can) return fail(PSX_ECUDA, "device %d cannot access peer %d", device, peer);
    PSX_DEVICE(device);
    cudaError_t e = cudaDeviceEnablePeerAccess(peer, 0);
    if (e == cudaErrorPeerAccessAlreadyEnabled) {
        cudaGetLastError();
        return PSX_OK;
    }
    if (e != cudaSuccess) return fail(PSX_ECUDA, "cudaDeviceEnablePeerAccess(%d->%d): %s", device, peer, cudaGetErrorString(e));
    return PSX_OK;
}

inline int grid_for(size_t work_items, int threads, int sm_count, int ctas_per_sm)
{
    size_t need = (work_items + threads - 1) / threads;
    size_t cap = (size_t)sm_count * ctas_per_sm;
    if (need < 1) need = 1;
    return (int)(need < cap ? need : cap);
}

#define LAUNCH_CHECK()                                                              \
    do {                                                                            \
        cudaError_t e_ = cudaGetLastError();                                        \
        if (e_ != cudaSuccess)                                                      \
            return fail(PSX_ECUDA, "kernel launch failed: %s (%s:%d)",              \
                        cudaGetErrorString(e_), __FILE__, __LINE__);                \
        g_launches.fetch_add(1, std::memory_order_relaxed);                         \
    } while (0)

// dst/src element types resolved at run time -> the four k_copy instances
int launch_copy(void *dst, int dst_t, const void *src, int src_t, uint64_t n, int sm_count,
                unsigned int *ticket, unsigned int *flag, uint32_t seq, cudaStream_t st,
                unsigned int *arrivals = nullptr, unsigned int *stamp_word = nullptr,
                uint32_t stamp = 0)
{
    if (n == 0 && flag == nullptr) return PSX_OK;
    const size_t sb = src_t == PSX_BF16 ? 2 : 4, db = dst_t == PSX_BF16 ? 2 : 4;
    // 4-element vectors: f32 needs 16 B alignment, bf16 8 B
    const int vec_ok = (((uintptr_t)src % (4 * sb)) == 0) && (((uintptr_t)dst % (4 * db)) == 0);
    const size_t items = vec_ok ? ((n >> 2) + kCopyUnroll - 1) / kCopyUnroll : n;
    const int grid = grid_for(items ? items : 1, kCopyThreads, sm_count, 8);
#define PSX_COPY(S, D)                                                                        \
    k_copy<S, D><<<grid, kCopyThreads, 0, st>>>((D *)dst, (const S *)src, (size_t)n, vec_ok, \
                                                 ticket, flag, arrivals, seq, stamp_word, stamp)
    if (src_t == PSX_F32 && dst_t == PSX_F32) PSX_COPY(float, float);
    else if (src_t == PSX_F32 && dst_t == PSX_BF16) PSX_COPY(float, __nv_bfloat16);
    else if (src_t == PSX_BF16 && dst_t == PSX_F32) PSX_COPY(__nv_bfloat16, float);
    else if (src_t == PSX_BF16 && dst_t == PSX_BF16) PSX_COPY(__nv_bfloat16, __nv_bfloat16);
    else return fail(PSX_EINVAL, "unknown dtype %d/%d", src_t, dst_t);
#undef PSX_COPY
    LAUNCH_CHECK();
    return PSX_OK;
}

// A launch covers elements [range.off, range.off + range.n) of the shard (multiples
// of 4); finish = 0 keeps the round open (no beta-power / step / apply_seq update).
struct ApplyRange {
    size_t off, n;
    int finish;
    unsigned int consume = 0;   // arrivals to take off the counter (counted rendez-vous)
    int divisor = 0;            // SYNC_MEAN denominator; 0 = the slot count
};

template <int OPT, int MODE, bool SCATTER, typename SRC>
void launch_apply_t(Shard *s, SRC src, int count, const PeerSet &peers, cudaStream_t st,
                    const ApplyRange &r)
{
    const size_t n4 = r.n / 4;
    const int grid = grid_for(n4 ? n4 : 1, kApplyThreads, s->sm_count, 3);
    k_apply<OPT, MODE, SCATTER, SRC><<<grid, kApplyThreads, 0, st>>>(
        s->hdr(), (float4 *)(s->var() + r.off), (float4 *)(s->m() + r.off),
        (float4 *)(s->v() + r.off), src, count, n4, peers, r.finish, r.consume,
        r.divisor ? r.divisor : count);
}

template <bool SCATTER, typename SRC>
int launch_apply(Shard *s, int mode, SRC src, int count, const PeerSet &peers, cudaStream_t st,
                 ApplyRange r = ApplyRange{0, 0, 1, 0, 0})
{
    if (r.n == 0 && r.off == 0) r.n = s->lay.nelem_pad;
#define PSX_AP(O, M) launch_apply_t<O, M, SCATTER, SRC>(s, src, count, peers, st, r)
#define PSX_AP3(O)                                                                            \
    if (mode == PSX_MODE_ASYNC_ORDERED) PSX_AP(O, PSX_MODE_ASYNC_ORDERED);                    \
    else if (mode == PSX_MODE_SUM) PSX_AP(O, PSX_MODE_SUM);                                   \
    else if (mode == PSX_MODE_SYNC_MEAN) PSX_AP(O, PSX_MODE_SYNC_MEAN);                       \
    else return fail(PSX_EINVAL, "unknown optimizer/mode %d/%d", opt, mode)
    const int opt = s->lay.opt;
    if (opt == PSX_OPT_SGD) { PSX_AP3(PSX_OPT_SGD); }
    else if (opt == PSX_OPT_ADAM) { PSX_AP3(PSX_OPT_ADAM); }
    else if (opt == PSX_OPT_MOMENTUM) { PSX_AP3(PSX_OPT_MOMENTUM); }
    else if (opt == PSX_OPT_ADAGRAD) { PSX_AP3(PSX_OPT_ADAGRAD); }
    else if (opt == PSX_OPT_RMSPROP) { PSX_AP3(PSX_OPT_RMSPROP); }
    else return fail(PSX_EINVAL, "unknown optimizer/mode %d/%d", opt, mode);
#undef PSX_AP3
#undef PSX_AP
    LAUNCH_CHECK();
    return PSX_OK;
}

struct Shard;
int launch_round_mc(Shard *s, int mode, const PeerSet &peers, cudaStream_t st, const ApplyRange &r);

void fill_mirrors(Shard *s, PeerSet *p)
{
    p->n_mirror = 0;
    p->n_param = 0;
    p->n_mailbox = 0;
    for (int c = 0; c < PSX_MAX_SLOTS; ++c) {
        if (s->mirror[c]) p->mirror[p->n_mirror++] = s->mirror[c];
        if (s->mailbox[c]) p->mailbox[p->n_mailbox++] = s->mailbox[c];
    }
}

int launch_round_mc(Shard *s, int mode, const PeerSet &peers, cudaStream_t st, const ApplyRange &r)
{
    const size_t n4 = r.n / 4;
    const size_t tile = (size_t)kMcThreads * PSX_MC_UNROLL;
    const size_t tiles = (n4 + tile - 1) / tile;
    const size_t cap = (size_t)s->sm_count * PSX_APPLY_MIN_CTAS;
    const int grid = (int)(tiles < 1 ? 1 : (tiles < cap ? tiles : cap));
#define PSX_MC(O, M)                                                                          \
    k_round_mc<O, M, PSX_MC_UNROLL><<<grid, kMcThreads, 0, st>>>(                             \
        s->hdr(), (float4 *)(s->var() + r.off), (float4 *)(s->m() + r.off),                   \
        (float4 *)(s->v() + r.off), s->mc_grad + r.off, s->mc_param + r.off, n4, peers,       \
        r.consume, r.divisor)
    const int opt = s->lay.opt;
#define PSX_MC2(O)                                                                            \
    if (mode == PSX_MODE_SUM) PSX_MC(O, PSX_MODE_SUM);                                        \
    else if (mode == PSX_MODE_SYNC_MEAN) PSX_MC(O, PSX_MODE_SYNC_MEAN);                       \
    else return fail(PSX_EINVAL, "the NVLS round supports SUM / SYNC_MEAN (optimizer/mode %d/%d)", opt, mode)
    if (opt == PSX_OPT_SGD) { PSX_MC2(PSX_OPT_SGD); }
    else if (opt == PSX_OPT_ADAM) { PSX_MC2(PSX_OPT_ADAM); }
    else if (opt == PSX_OPT_MOMENTUM) { PSX_MC2(PSX_OPT_MOMENTUM); }
    else if (opt == PSX_OPT_ADAGRAD) { PSX_MC2(PSX_OPT_ADAGRAD); }
    else if (opt == PSX_OPT_RMSPROP) { PSX_MC2(PSX_OPT_RMSPROP); }
    else return fail(PSX_EINVAL, "the NVLS round supports SUM / SYNC_MEAN (optimizer/mode %d/%d)", opt, mode);
#undef PSX_MC2
#undef PSX_MC
    LAUNCH_CHECK();
    return PSX_OK;
}

// ------------------------------------------------- request-free serving ----
// One host thread per served shard.  It POLLS the shard's arrival counter (a
// 4-byte device->host copy on the serving stream, ~6 us) and, when pushes have
// arrived, launches  k_pick ; k_apply<.., PickSrc>  on that stream.
//
// Why not pre-enqueued cuStreamWaitValue32(arrivals >= 1) iterations (the first
// implementation): a stream blocked in a wait-value holds its hardware channel,
// and CUDA multiplexes all streams of a process onto a few channels
// (CUDA_DEVICE_MAX_CONNECTIONS, 8 by default).  Work submitted LATER on another
// stream that aliases to the same channel -- the push that would satisfy the
// wait when worker and PS share a process, or the accessor / stop path inside the
// PS process -- queues up BEHIND the wait and never runs: a deadlock that depends
// on how many streams the process happens to have created (it took a whole test
// run down, profiles/r23).  Every stream wait this library still issues is
// submitted after the work it waits for (or waits for another process), so
// submission order is always a valid execution order.
struct Server {
    std::thread th;
    std::atomic<bool> stop{false};
    cudaStream_t stream = nullptr;
    int mode = PSX_MODE_ASYNC_ORDERED, aggregate = 1, idle_sleep_us = 0;
    std::atomic<uint64_t> iterations{0};
    std::atomic<int> error{0};
    char errmsg[256] = "";
};

int serve_iteration(Shard *s, Server *sv)
{
    const int n_slots = s->lay.n_slots;
    if (sv->mode == PSX_MODE_ASYNC_ORDERED)
        k_pick<PSX_MODE_ASYNC_ORDERED><<<1, 32, 0, sv->stream>>>(s->hdr(), n_slots, 1);
    else
        k_pick<PSX_MODE_SYNC_MEAN><<<1, 32, 0, sv->stream>>>(s->hdr(), n_slots, sv->aggregate);
    LAUNCH_CHECK();
    PeerSet peers;
    memset(&peers, 0, sizeof(peers));
    const ApplyRange r{0, (size_t)s->lay.nelem_pad, 1, 0, 0};
    if (s->lay.wire == PSX_F32) {
        PickSrc<float> src{(const float *)s->slot(0), (size_t)s->lay.nelem_pad, nullptr};
        return launch_apply<false>(s, sv->mode, src, 0, peers, sv->stream, r);
    }
    PickSrc<__nv_bfloat16> src{(const __nv_bfloat16 *)s->slot(0), (size_t)s->lay.nelem_pad, nullptr};
    return launch_apply<false>(s, sv->mode, src, 0, peers, sv->stream, r);
}

void serve_main(Shard *s, Server *sv)
{
    cudaSetDevice(s->device);
    unsigned int *seen = nullptr;                 // pinned landing word of the poll
    cudaError_t e = cudaHostAlloc((void **)&seen, sizeof(unsigned int), cudaHostAllocDefault);
    uint64_t it = 0;
    int idle = 0;
    while (e == cudaSuccess && !sv->stop.load()) {
        // ordered behind the previous iteration's kernels: reads the counter AFTER
        // that pick took its pushes off
        e = cudaMemcpyAsync(seen, &s->hdr()->arrivals, sizeof(unsigned int), cudaMemcpyDeviceToHost,
                            sv->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(sv->stream);
        if (e != cudaSuccess) break;
        if ((int)*seen < 1) {                     // signed: a pick may run ahead of a counter bump
            if (sv->idle_sleep_us > 0 && ++idle > 64) usleep((useconds_t)sv->idle_sleep_us);
            continue;
        }
        idle = 0;
        int rc = serve_iteration(s, sv);
        if (rc) {
            snprintf(sv->errmsg, sizeof(sv->errmsg), "%.250s", g_err);
            sv->error.store(rc);
            break;
        }
        sv->iterations.store(++it);
    }
    cudaError_t e2 = cudaStreamSynchronize(sv->stream);
    if (e == cudaSuccess) e = e2;
    if (e != cudaSuccess && sv->error.load() == 0) {
        snprintf(sv->errmsg, sizeof(sv->errmsg), "serving stream: %s", cudaGetErrorString(e));
        sv->error.store(PSX_ECUDA);
    }
    if (seen) cudaFreeHost(seen);
}

int serve_start_impl(Shard *s, int mode, int aggregate, int idle_sleep_us)
{
    if (s->server) return fail(PSX_ESTATE, "shard is already being served");
    if (s->lay.n_slots < 1) return fail(PSX_ESTATE, "serving needs landing slots (n_slots >= 1)");
    if (mode != PSX_MODE_ASYNC_ORDERED && mode != PSX_MODE_SYNC_MEAN)
        return fail(PSX_EINVAL, "serve mode must be ASYNC_ORDERED or SYNC_MEAN");
    if (mode == PSX_MODE_SYNC_MEAN && (aggregate < 1 || aggregate > s->lay.n_slots))
        return fail(PSX_EINVAL, "replicas_to_aggregate %d outside 1..%d", aggregate, s->lay.n_slots);
    if (idle_sleep_us < 0) idle_sleep_us = 0;
    PSX_DEVICE(s->device);
    Server *sv = new Server();
    sv->mode = mode;
    sv->aggregate = aggregate;
    sv->idle_sleep_us = idle_sleep_us;
    cudaError_t e = cudaStreamCreateWithFlags(&sv->stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) {
        delete sv;
        return fail(PSX_ECUDA, "creating the serving stream: %s", cudaGetErrorString(e));
    }
    s->server = sv;
    sv->th = std::thread(serve_main, s, sv);
    return PSX_OK;
}

// Stops the loop and leaves the shard quiescent (the thread finishes the iteration
// it is in).  Pushes that arrive while stopped stay flagged and counted for the
// next psx_serve_start.
int serve_stop_impl(Shard *s, int *mode, int *aggregate, int *idle_sleep_us)
{
    Server *sv = s->server;
    if (!sv) return PSX_OK;
    sv->stop.store(true);
    sv->th.join();
    {
        DeviceGuard g(s->device);
        cudaStreamDestroy(sv->stream);
    }
    if (mode) *mode = sv->mode;
    if (aggregate) *aggregate = sv->aggregate;
    if (idle_sleep_us) *idle_sleep_us = sv->idle_sleep_us;
    int err = sv->error.load();
    char msg[256];
    snprintf(msg, sizeof(msg), "%s", sv->errmsg);
    s->server = nullptr;
    delete sv;
    if (err) return fail(err, "serving loop failed: %s", msg);
    return PSX_OK;
}

// Host accessors pause the serving loop for their duration: one consistent view of
// var / m / v / state, and no apply is launched under a host copy.
struct ServePause {
    Shard *s;
    std::unique_lock<std::recursive_mutex> lk;    // held for the accessor's whole duration
    bool was = false;
    int mode = 0, aggregate = 1, depth = 0, rc = PSX_OK;
    explicit ServePause(Shard *sh) : s(sh), lk(sh->serve_mu)
    {
        if (s->server) {
            was = true;
            rc = serve_stop_impl(s, &mode, &aggregate, &depth);
        }
    }
    ~ServePause()
    {
        if (was && rc == PSX_OK) serve_start_impl(s, mode, aggregate, depth);
    }
};
#define PSX_PAUSE(shard)              \
    ServePause pause_(shard);         \
    if (pause_.rc) return pause_.rc

int wait_slots(Shard *s, int first, int count, uint32_t wait_seq, void *stream)
{
    if (wait_seq == 0) return PSX_OK;
    for (int k = 0; k < count; ++k) {
        int rc = stream_wait_geq(stream, &s->hdr()->slot_seq[first + k], wait_seq);
        if (rc) return rc;
    }
    return PSX_OK;
}

int check_range(int first, int count, int n_slots)
{
    if (count < 1 || first < 0 || first + count > n_slots || count > PSX_MAX_SLOTS)
        return fail(PSX_EINVAL, "slot range [%d, %d) outside the shard's %d slots", first,
                    first + count, n_slots);
    return PSX_OK;
}

}  // namespace

// =============================================================== C ABI =======
extern "C" {

int psx_abi_version(void) { return PSX_ABI_VERSION; }

const char *psx_last_error(void) { return g_err; }

uint64_t psx_launch_count(void) { return g_launches.load(); }

int psx_device_count(int *out_n)
{
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (out_n) *out_n = (e == cudaSuccess) ? n : 0;
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(PSX_ECUDA, "cudaGetDeviceCount: %s", cudaGetErrorString(e));
    }
    if (n == 0) return fail(PSX_ECUDA, "no CUDA device visible");
    return PSX_OK;
}

int psx_init(int device)
{
    int n = 0;
    int rc = psx_device_count(&n);
    if (rc) return rc;
    if (device < 0 || device >= n) return fail(PSX_EINVAL, "device %d out of range [0,%d)", device, n);
    CU_TRY(cudaSetDevice(device));  // sticks: this is the process's device from now on
    CU_TRY(cudaFree(0));            // force the primary context
    return resolve_memops();
}

int psx_enable_peer(int device, int peer) { return enable_peer(device, peer); }

// ------------------------------------------------------------------ PS side --
int psx_shard_create(int device, uint64_t nelem, int opt, const float *hyper, int n_slots,
                     int wire_dtype, uint64_t *out_id)
{
    if (!out_id || !hyper) return fail(PSX_EINVAL, "null argument");
    if (nelem == 0) return fail(PSX_EINVAL, "empty shard");
    if (state_arrays(opt) < 0) return fail(PSX_EINVAL, "unknown optimizer %d", opt);
    if (opt == PSX_OPT_ADAGRAD && !(hyper[1] > 0.0f))
        return fail(PSX_EINVAL, "Adagrad initial_accumulator_value must be > 0 (got %g)", (double)hyper[1]);
    if (n_slots < 0 || n_slots > PSX_MAX_SLOTS) return fail(PSX_EINVAL, "n_slots %d not in [0,%d]", n_slots, PSX_MAX_SLOTS);
    if (wire_dtype != PSX_F32 && wire_dtype != PSX_BF16) return fail(PSX_EINVAL, "unknown wire dtype %d", wire_dtype);
    PSX_DEVICE(device);
    Shard *s = new Shard();
    s->device = device;
    s->lay.nelem = nelem;
    s->lay.nelem_pad = (nelem + kPadElems - 1) / kPadElems * kPadElems;
    s->lay.opt = opt;
    s->lay.n_slots = n_slots;
    s->lay.wire = wire_dtype;
    s->sm_count = sm_count_of(device);
    void *p = nullptr;
    cudaError_t e = cudaMalloc(&p, s->lay.total());
    if (e != cudaSuccess) {
        size_t total = s->lay.total();
        delete s;
        cudaGetLastError();
        return fail(e == cudaErrorMemoryAllocation ? PSX_ENOMEM : PSX_ECUDA,
                    "cudaMalloc(%zu bytes) for shard: %s", total, cudaGetErrorString(e));
    }
    s->base = (char *)p;
    e = cudaMemset(p, 0, s->lay.total());
    ShardHeader h;
    memset(&h, 0, sizeof(h));
    h.magic = kMagic;
    h.abi = PSX_ABI_VERSION;
    h.lr = hyper[0];
    h.b1 = hyper[1];
    h.b2 = hyper[2];
    h.eps = hyper[3];
    h.b1p = hyper[1];  // powers start at beta (AdamOptimizer._create_slots)
    h.b2p = hyper[2];
    if (e == cudaSuccess) e = cudaMemcpy(p, &h, sizeof(h), cudaMemcpyHostToDevice);
    // accumulators that do not start at zero: Adagrad's at initial_accumulator_value,
    // RMSProp's ms at 1 (TF's `rms` slot initializer); padding included
    const float m0 = opt == PSX_OPT_ADAGRAD ? hyper[1] : opt == PSX_OPT_RMSPROP ? 1.0f : 0.0f;
    if (e == cudaSuccess && m0 != 0.0f) {
        const size_t n4 = s->lay.nelem_pad / 4;
        k_fill<<<grid_for(n4, kCopyThreads, s->sm_count, 8), kCopyThreads>>>((float4 *)s->m(), m0, n4);
        e = cudaGetLastError();
        if (e == cudaSuccess) e = cudaDeviceSynchronize();
        if (e == cudaSuccess) g_launches.fetch_add(1, std::memory_order_relaxed);
    }
    if (e != cudaSuccess) {
        cudaFree(p);
        delete s;
        return fail(PSX_ECUDA, "initialising shard: %s", cudaGetErrorString(e));
    }
    uint64_t id = g_next_id.fetch_add(1);
    {
        std::lock_guard<std::mutex> lk(g_mu);
        g_shards[id] = s;
    }
    *out_id = id;
    return PSX_OK;
}

int psx_shard_destroy(uint64_t id)
{
    Shard *s = nullptr;
    {
        std::lock_guard<std::mutex> lk(g_mu);
        auto it = g_shards.find(id);
        if (it == g_shards.end()) return fail(PSX_EINVAL, "unknown shard id %llu", (unsigned long long)id);
        s = it->second;
        g_shards.erase(it);
    }
    int src;
    {
        std::lock_guard<std::recursive_mutex> lk(s->serve_mu);
        src = serve_stop_impl(s, nullptr, nullptr, nullptr);
    }
    cudaError_t e = cudaSetDevice(s->device);
    if (e == cudaSuccess) e = cudaDeviceSynchronize();   // a failed kernel surfaces here
    for (int c = 0; c < PSX_MAX_SLOTS; ++c) {
        close_mapped(s->client_map[c]);
        close_mapped(s->mailbox_map[c]);
        close_mapped(s->bound[c].grad);
        close_mapped(s->bound[c].param);
    }
    cudaError_t e2 = cudaFree(s->base);
    delete s;
    if (e == cudaSuccess) e = e2;
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(PSX_ECUDA, "destroying shard %llu: %s", (unsigned long long)id, cudaGetErrorString(e));
    }
    return src;
}

int psx_shard_export(uint64_t id, void *out_handle)
{
    Shard *s = find(g_shards, id);
    if (!s || !out_handle) return fail(PSX_EINVAL, "unknown shard id or null handle");
    HandleBlob b;
    memset(&b, 0, sizeof(b));
    b.magic = kMagic;
    b.abi = PSX_ABI_VERSION;
    b.kind = KIND_SHARD;
    b.device = s->device;
    b.pid = (uint64_t)getpid();
    b.local_id = id;
    b.nelem = s->lay.nelem;
    b.nelem_pad = s->lay.nelem_pad;
    b.opt = s->lay.opt;
    b.n_slots = s->lay.n_slots;
    b.wire = s->lay.wire;
    PSX_DEVICE(s->device);
    CU_TRY(cudaIpcGetMemHandle(&b.ipc, s->base));
    memcpy(out_handle, &b, sizeof(b));
    return PSX_OK;
}

int psx_shard_set_hyper(uint64_t id, const float *hyper)
{
    Shard *s = find(g_shards, id);
    if (!s || !hyper) return fail(PSX_EINVAL, "unknown shard id or null hyper");
    PSX_PAUSE(s);
    PSX_DEVICE(s->device);
    CU_TRY(cudaDeviceSynchronize());   // not under a running apply
    CU_TRY(cudaMemcpy(&s->hdr()->lr, hyper, 4 * sizeof(float), cudaMemcpyHostToDevice));
    return PSX_OK;
}

static int region_of(Shard *s, int which, char **base, int *dtype)
{
    *dtype = PSX_F32;
    if (which == PSX_VAR) *base = (char *)s->var();
    else if (which == PSX_M && s->lay.n_state() >= 1) *base = (char *)s->m();
    else if (which == PSX_V && s->lay.n_state() >= 2) *base = (char *)s->v();
    else if (which >= PSX_SLOT0 && which < PSX_SLOT0 + s->lay.n_slots) {
        *base = s->slot(which - PSX_SLOT0);
        *dtype = s->lay.wire;
    } else
        return fail(PSX_EINVAL, "shard has no region %d", which);
    return PSX_OK;
}

int psx_set_values(uint64_t id, int which, const float *host, uint64_t off, uint64_t n)
{
    Shard *s = find(g_shards, id);
    if (!s) return fail(PSX_EINVAL, "unknown shard id");
    if (off + n > s->lay.nelem) return fail(PSX_EINVAL, "range [%llu,+%llu) outside shard of %llu", (unsigned long long)off, (unsigned long long)n, (unsigned long long)s->lay.nelem);
    char *base;
    int dt;
    int rc = region_of(s, which, &base, &dt);
    if (rc) return rc;
    if (n == 0) return PSX_OK;
    PSX_PAUSE(s);
    PSX_DEVICE(s->device);
    // synchronous by contract: kernels on non-blocking streams are not ordered
    // against the legacy stream's memcpy, so drain the device first
    CU_TRY(cudaDeviceSynchronize());
    if (dt == PSX_F32) {
        CU_TRY(cudaMemcpy(base + off * 4, host, n * 4, cudaMemcpyHostToDevice));
    } else {  // stage f32 on the device, cast with the push kernel
        void *tmp = nullptr;
        CU_TRY(cudaMalloc(&tmp, n * 4));
        cudaError_t e = cudaMemcpy(tmp, host, n * 4, cudaMemcpyHostToDevice);
        if (e == cudaSuccess) {
            rc = launch_copy(base + off * 2, PSX_BF16, tmp, PSX_F32, n, s->sm_count, nullptr, nullptr, 0, 0);
            e = cudaDeviceSynchronize();
        }
        cudaFree(tmp);
        if (rc) return rc;
        if (e != cudaSuccess) return fail(PSX_ECUDA, "set_values(bf16): %s", cudaGetErrorString(e));
    }
    return PSX_OK;
}

int psx_get_values(uint64_t id, int which, float *host, uint64_t off, uint64_t n)
{
    Shard *s = find(g_shards, id);
    if (!s) return fail(PSX_EINVAL, "unknown shard id");
    if (off + n > s->lay.nelem) return fail(PSX_EINVAL, "range outside shard");
    char *base;
    int dt;
    int rc = region_of(s, which, &base, &dt);
    if (rc) return rc;
    if (n == 0) return PSX_OK;
    PSX_PAUSE(s);
    PSX_DEVICE(s->device);
    CU_TRY(cudaDeviceSynchronize());
    if (dt == PSX_F32) {
        CU_TRY(cudaMemcpy(host, base + off * 4, n * 4, cudaMemcpyDeviceToHost));
    } else {
        void *tmp = nullptr;
        CU_TRY(cudaMalloc(&tmp, n * 4));
        rc = launch_copy(tmp, PSX_F32, base + off * 2, PSX_BF16, n, s->sm_count, nullptr, nullptr, 0, 0);
        cudaError_t e = cudaDeviceSynchronize();
        if (e == cudaSuccess) e = cudaMemcpy(host, tmp, n * 4, cudaMemcpyDeviceToHost);
        cudaFree(tmp);
        if (rc) return rc;
        if (e != cudaSuccess) return fail(PSX_ECUDA, "get_values(bf16): %s", cudaGetErrorString(e));
    }
    return PSX_OK;
}

int psx_get_state(uint64_t id, float *b1p, float *b2p, int64_t *step, uint32_t *apply_seq)
{
    Shard *s = find(g_shards, id);
    if (!s) return fail(PSX_EINVAL, "unknown shard id");
    PSX_PAUSE(s);
    PSX_DEVICE(s->device);
    CU_TRY(cudaDeviceSynchronize());
    ShardHeader h;
    CU_TRY(cudaMemcpy(&h, s->base, sizeof(h), cudaMemcpyDeviceToHost));
    if (b1p) *b1p = h.b1p;
    if (b2p) *b2p = h.b2p;
    if (step) *step = h.step;
    if (apply_seq) *apply_seq = h.apply_seq;
    return PSX_OK;
}

int psx_set_state(uint64_t id, float b1p, float b2p, int64_t step)
{
    Shard *s = find(g_shards, id);
    if (!s) return fail(PSX_EINVAL, "unknown shard id");
    PSX_PAUSE(s);
    PSX_DEVICE(s->device);
    CU_TRY(cudaDeviceSynchronize());
    ShardHeader h;
    CU_TRY(cudaMemcpy(&h, s->base, sizeof(h), cudaMemcpyDeviceToHost));
    h.b1p = b1p;
    h.b2p = b2p;
    h.step = step;
    CU_TRY(cudaMemcpy(s->base, &h, offsetof(ShardHeader, ticket), cudaMemcpyHostToDevice));
    return PSX_OK;
}

int psx_shard_ptr(uint64_t id, int which, void **out_dev_ptr)
{
    Shard *s = find(g_shards, id);
    if (!s || !out_dev_ptr) return fail(PSX_EINVAL, "unknown shard id or null out pointer");
    char *base;
    int dt;
    int rc = region_of(s, which, &base, &dt);
    if (rc) return rc;
    *out_dev_ptr = base;
    return PSX_OK;
}

int psx_apply_range(uint64_t id, int mode, int first_slot, int count, uint64_t elem_off,
                    uint64_t elem_n, int finish, uint32_t wait_seq, void *stream)
{
    Shard *s = find(g_shards, id);
    if (!s) return fail(PSX_EINVAL, "unknown shard id");
    int rc = check_range(first_slot, count, s->lay.n_slots);
    if (rc) return rc;
    if (elem_n == 0) {                      // whole shard
        elem_off = 0;
        elem_n = s->lay.nelem_pad;
    } else {
        if (elem_off % 4) return fail(PSX_EINVAL, "elem_off must be a multiple of 4");
        if (elem_off + elem_n > s->lay.nelem_pad)
            return fail(PSX_EINVAL, "apply range [%llu,+%llu) outside the shard", (unsigned long long)elem_off, (unsigned long long)elem_n);
        if (elem_n % 4 && elem_off + elem_n < s->lay.nelem)
            return fail(PSX_EINVAL, "an inner apply range must be a multiple of 4 elements");
        elem_n = (elem_n + 3) / 4 * 4;      // the padding up to nelem_pad is always allocated
        if (elem_off + elem_n > s->lay.nelem_pad) elem_n = s->lay.nelem_pad - elem_off;
    }
    PSX_DEVICE(s->device);
    rc = wait_slots(s, first_slot, count, wait_seq, stream);
    if (rc) return rc;
    PeerSet peers;
    memset(&peers, 0, sizeof(peers));
    fill_mirrors(s, &peers);
    const ApplyRange r{(size_t)elem_off, (size_t)elem_n, finish ? 1 : 0, 0, 0};
    if (s->lay.wire == PSX_F32) {
        SlotSrc<float> src{(const float *)s->slot(0) + elem_off, (size_t)s->lay.nelem_pad, first_slot};
        return launch_apply<false>(s, mode, src, count, peers, (cudaStream_t)stream, r);
    }
    SlotSrc<__nv_bfloat16> src{(const __nv_bfloat16 *)s->slot(0) + elem_off, (size_t)s->lay.nelem_pad, first_slot};
    return launch_apply<false>(s, mode, src, count, peers, (cudaStream_t)stream, r);
}

int psx_apply(uint64_t id, int mode, int first_slot, int count, uint32_t wait_seq, void *stream)
{
    return psx_apply_range(id, mode, first_slot, count, 0, 0, 1, wait_seq, stream);
}

int psx_apply_counted(uint64_t id, int mode, int first_slot, int count, void *stream)
{
    Shard *s = find(g_shards, id);
    if (!s) return fail(PSX_EINVAL, "unknown shard id");
    int rc = check_range(first_slot, count, s->lay.n_slots);
    if (rc) return rc;
    PSX_DEVICE(s->device);
    rc = stream_wait_geq(stream, &s->hdr()->arrivals, (uint32_t)count);
    if (rc) return rc;
    PeerSet peers;
    memset(&peers, 0, sizeof(peers));
    fill_mirrors(s, &peers);
    const ApplyRange r{0, (size_t)s->lay.nelem_pad, 1, (unsigned int)count, 0};
    if (s->lay.wire == PSX_F32) {
        SlotSrc<float> src{(const float *)s->slot(0), (size_t)s->lay.nelem_pad, first_slot};
        return launch_apply<false>(s, mode, src, count, peers, (cudaStream_t)stream, r);
    }
    SlotSrc<__nv_bfloat16> src{(const __nv_bfloat16 *)s->slot(0), (size_t)s->lay.nelem_pad, first_slot};
    return launch_apply<false>(s, mode, src, count, peers, (cudaStream_t)stream, r);
}

int psx_wait_slots(uint64_t id, int first_slot, int count, uint32_t wait_seq, void *stream)
{
    Shard *s = find(g_shards, id);
    if (!s) return fail(PSX_EINVAL, "unknown shard id");
    int rc = check_range(first_slot, count, PSX_MAX_SLOTS);
    if (rc) return rc;
    PSX_DEVICE(s->device);
    return wait_slots(s, first_slot, count, wait_seq, stream);
}

int psx_shard_register_client(uint64_t shard_id, int slot, const void *client_handle)
{
    Shard *s = find(g_shards, shard_id);
    if (!s) return fail(PSX_EINVAL, "unknown shard id");
    if (slot < 0 || slot >= PSX_MAX_SLOTS) return fail(PSX_EINVAL, "slot %d out of range", slot);
    HandleBlob b;
    int rc = check_blob(client_handle, KIND_CLIENT, &b);
    if (rc) return rc;
    if (s->mirror[slot]) {   // re-registration (a revived worker): nothing in flight may
        PSX_PAUSE(s);            // still hold the old mapping
        PSX_DEVICE(s->device);
        CU_TRY(cudaDeviceSynchronize());
        s->mirror[slot] = nullptr;
        unsigned long long zero = 0;
        CU_TRY(cudaMemcpy(&s->hdr()->client_block[slot], &zero, sizeof(zero), cudaMemcpyHostToDevice));
        close_mapped(s->client_map[slot]);
    }
    rc = open_blob(b, s->device, &s->client_map[slot]);
    if (rc) return rc;
    s->mirror[slot] = &((ClientBlock *)s->client_map[slot].base)->applied;
    {   // the served epilogue finds the block through the header, at run time
        PSX_DEVICE(s->device);
        unsigned long long addr = (unsigned long long)(uintptr_t)s->client_map[slot].base;
        CU_TRY(cudaMemcpy(&s->hdr()->client_block[slot], &addr, sizeof(addr), cudaMemcpyHostToDevice));
    }
    return PSX_OK;
}

/* Detach worker `slot` from the shard: drains the shard's device (no apply may be
 * in flight that still publishes into the worker's block), then unmaps the
 * worker's client block, mailbox and bound buffers.  The worker calls this (via
 * its PS endpoint) BEFORE it frees those objects -- a PS that kept publishing
 * into freed peer memory would take its own context down. */
int psx_shard_unregister_client(uint64_t shard_id, int slot)
{
    Shard *s = find(g_shards, shard_id);
    if (!s) return fail(PSX_EINVAL, "unknown shard id");
    if (slot < 0 || slot >= PSX_MAX_SLOTS) return fail(PSX_EINVAL, "slot %d out of range", slot);
    PSX_PAUSE(s);
    PSX_DEVICE(s->device);
    CU_TRY(cudaDeviceSynchronize());
    s->mirror[slot] = nullptr;
    unsigned long long zero = 0;
    CU_TRY(cudaMemcpy(&s->hdr()->client_block[slot], &zero, sizeof(zero), cudaMemcpyHostToDevice));
    close_mapped(s->client_map[slot]);
    s->mailbox[slot] = nullptr;
    close_mapped(s->mailbox_map[slot]);
    if (s->bound[slot].valid) {
        close_mapped(s->bound[slot].grad);
        close_mapped(s->bound[slot].param);
        s->bound[slot].valid = false;
    }
    return PSX_OK;
}

// -------------------------------------------------------------- worker side --
int psx_shard_open(const void *handle, int device, int slot, uint64_t *out_id)
{
    if (!out_id) return fail(PSX_EINVAL, "null out id");
    HandleBlob b;
    int rc = check_blob(handle, KIND_SHARD, &b);
    if (rc) return rc;
    if (slot < 0 || slot >= PSX_MAX_SLOTS || (b.n_slots > 0 && slot >= b.n_slots))
        return fail(PSX_EINVAL, "slot %d outside the shard's %d slots", slot,
                    b.n_slots > 0 ? b.n_slots : PSX_MAX_SLOTS);
    Client *c = new Client();
    c->device = device;
    c->slot = slot;
    c->lay.nelem = b.nelem;
    c->lay.nelem_pad = b.nelem_pad;
    c->lay.opt = b.opt;
    c->lay.n_slots = b.n_slots;
    c->lay.wire = b.wire;
    c->sm_count = sm_count_of(device);
    rc = open_blob(b, device, &c->shard);
    if (rc) {
        delete c;
        return rc;
    }
    DeviceGuard guard(device);
    cudaError_t e = guard.err;
    void *blk = nullptr;
    if (e == cudaSuccess) e = cudaMalloc(&blk, sizeof(ClientBlock));
    if (e == cudaSuccess) e = cudaMemset(blk, 0, sizeof(ClientBlock));
    if (e != cudaSuccess) {
        close_mapped(c->shard);
        delete c;
        return fail(PSX_ECUDA, "allocating client block: %s", cudaGetErrorString(e));
    }
    c->block = (ClientBlock *)blk;
    uint64_t id = g_next_id.fetch_add(1);
    {
        std::lock_guard<std::mutex> lk(g_mu);
        g_clients[id] = c;
    }
    *out_id = id;
    return PSX_OK;
}

int psx_shard_close(uint64_t id)
{
    Client *c = nullptr;
    {
        std::lock_guard<std::mutex> lk(g_mu);
        auto it = g_clients.find(id);
        if (it == g_clients.end()) return fail(PSX_EINVAL, "unknown client id");
        c = it->second;
        g_clients.erase(it);
    }
    cudaError_t e = cudaSetDevice(c->device);
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    close_mapped(c->shard);
    if (c->poll_stream) cudaStreamDestroy(c->poll_stream);
    cudaError_t e2 = cudaFree(c->block);
    delete c;
    if (e == cudaSuccess) e = e2;
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(PSX_ECUDA, "closing client %llu: %s", (unsigned long long)id, cudaGetErrorString(e));
    }
    return PSX_OK;
}

int psx_client_export(uint64_t client_id, void *out_handle)
{
    Client *c = find(g_clients, client_id);
    if (!c || !out_handle) return fail(PSX_EINVAL, "unknown client id or null handle");
    HandleBlob b;
    memset(&b, 0, sizeof(b));
    b.magic = kMagic;
    b.abi = PSX_ABI_VERSION;
    b.kind = KIND_CLIENT;
    b.device = c->device;
    b.pid = (uint64_t)getpid();
    b.local_id = client_id;
    PSX_DEVICE(c->device);
    CU_TRY(cudaIpcGetMemHandle(&b.ipc, c->block));
    memcpy(out_handle, &b, sizeof(b));
    return PSX_OK;
}

int psx_push(uint64_t client_id, const void *grad_dev, uint64_t off, uint64_t n, int src_dtype,
             uint32_t seq, void *stream)
{
    Client *c = find(g_clients, client_id);
    if (!c) return fail(PSX_EINVAL, "unknown client id");
    if (c->lay.n_slots == 0) return fail(PSX_ESTATE, "shard was created without gradient slots");
    if (off + n > c->lay.nelem) return fail(PSX_EINVAL, "push range [%llu,+%llu) outside shard of %llu", (unsigned long long)off, (unsigned long long)n, (unsigned long long)c->lay.nelem);
    if (n && !grad_dev) return fail(PSX_EINVAL, "null gradient pointer");
    PSX_DEVICE(c->device);
    char *dst = c->my_slot() + off * c->lay.wire_bytes();
    unsigned int *flag = seq ? &c->hdr()->slot_seq[c->slot] : nullptr;
    return launch_copy(dst, c->lay.wire, grad_dev, src_dtype, n, c->sm_count, &c->block->ticket,
                       flag, seq, (cudaStream_t)stream, seq ? &c->hdr()->arrivals : nullptr);
}

int psx_pull(uint64_t client_id, void *param_dev, uint64_t off, uint64_t n, int out_dtype,
             uint32_t wait_seq, void *stream)
{
    Client *c = find(g_clients, client_id);
    if (!c) return fail(PSX_EINVAL, "unknown client id");
    if (off + n > c->lay.nelem) return fail(PSX_EINVAL, "pull range outside shard");
    if (n && !param_dev) return fail(PSX_EINVAL, "null parameter pointer");
    PSX_DEVICE(c->device);
    if (wait_seq) {
        int rc = stream_wait_geq(stream, &c->block->applied, wait_seq);
        if (rc) return rc;
    }
    if (n == 0) return PSX_OK;
    return launch_copy(param_dev, out_dtype, c->var() + off, PSX_F32, n, c->sm_count, nullptr,
                       nullptr, 0, (cudaStream_t)stream);
}

static int signal_impl(const uint64_t *client_ids, int n, uint32_t seq, uint64_t mailbox_id,
                       uint32_t consume, void *stream)
{
    if (!client_ids || n < 1 || n > kMaxSignal)
        return fail(PSX_EINVAL, "psx_signal_many takes 1..%d clients", kMaxSignal);
    SignalSet set;
    memset(&set, 0, sizeof(set));
    set.n = n;
    if (mailbox_id) {
        Mailbox *m = find(g_mailboxes, mailbox_id);
        if (!m) return fail(PSX_EINVAL, "unknown mailbox id");
        set.mailbox = m->counter;
        set.consume = consume;
    }
    int device = -1;
    for (int i = 0; i < n; ++i) {
        Client *c = find(g_clients, client_ids[i]);
        if (!c) return fail(PSX_EINVAL, "unknown client id (entry %d)", i);
        if (device < 0) device = c->device;
        if (c->device != device) return fail(PSX_EINVAL, "clients of one signal must share a device");
        set.flag[i] = &c->hdr()->slot_seq[c->slot];
        set.arrivals[i] = &c->hdr()->arrivals;
    }
    PSX_DEVICE(device);
    k_signal<<<1, kMaxSignal, 0, (cudaStream_t)stream>>>(set, seq);
    LAUNCH_CHECK();
    return PSX_OK;
}

int psx_signal_many(const uint64_t *client_ids, int n, uint32_t seq, void *stream)
{
    return signal_impl(client_ids, n, seq, 0, 0, stream);
}

int psx_signal_counted(const uint64_t *client_ids, int n, uint32_t seq, uint64_t mailbox_id,
                       uint32_t consume, void *stream)
{
    return signal_impl(client_ids, n, seq, mailbox_id, consume, stream);
}

int psx_signal(uint64_t client_id, uint32_t seq, void *stream)
{
    return psx_signal_many(&client_id, 1, seq, stream);
}

int psx_mailbox_set(uint64_t id, uint32_t value)
{
    Mailbox *m = find(g_mailboxes, id);
    if (!m) return fail(PSX_EINVAL, "unknown mailbox id");
    PSX_DEVICE(m->device);
    CU_TRY(cudaDeviceSynchronize());
    CU_TRY(cudaMemcpy(m->counter, &value, sizeof(value), cudaMemcpyHostToDevice));
    return PSX_OK;
}

int psx_mailbox_consume(uint64_t id, uint32_t n, void *stream)
{
    Mailbox *m = find(g_mailboxes, id);
    if (!m) return fail(PSX_EINVAL, "unknown mailbox id");
    PSX_DEVICE(m->device);
    k_consume<<<1, 1, 0, (cudaStream_t)stream>>>(m->counter, n);
    LAUNCH_CHECK();
    return PSX_OK;
}

int psx_wait_arrivals(uint64_t shard_id, uint32_t target, void *stream)
{
    Shard *s = find(g_shards, shard_id);
    if (!s) return fail(PSX_EINVAL, "unknown shard id");
    PSX_DEVICE(s->device);
    return stream_wait_geq(stream, &s->hdr()->arrivals, target);
}

int psx_mailbox_create(int device, uint64_t *out_id)
{
    if (!out_id) return fail(PSX_EINVAL, "null out id");
    PSX_DEVICE(device);
    void *p = nullptr;
    CU_TRY(cudaMalloc(&p, 256));
    CU_TRY(cudaMemset(p, 0, 256));
    Mailbox *m = new Mailbox();
    m->device = device;
    m->counter = (unsigned int *)p;
    uint64_t id = g_next_id.fetch_add(1);
    {
        std::lock_guard<std::mutex> lk(g_mu);
        g_mailboxes[id] = m;
    }
    *out_id = id;
    return PSX_OK;
}

int psx_mailbox_export(uint64_t id, void *out_handle)
{
    Mailbox *m = find(g_mailboxes, id);
    if (!m || !out_handle) return fail(PSX_EINVAL, "unknown mailbox id or null handle");
    HandleBlob b;
    memset(&b, 0, sizeof(b));
    b.magic = kMagic;
    b.abi = PSX_ABI_VERSION;
    b.kind = KIND_MAILBOX;
    b.device = m->device;
    b.pid = (uint64_t)getpid();
    b.local_id = id;
    PSX_DEVICE(m->device);
    CU_TRY(cudaIpcGetMemHandle(&b.ipc, m->counter));
    memcpy(out_handle, &b, sizeof(b));
    return PSX_OK;
}

int psx_mailbox_destroy(uint64_t id)
{
    Mailbox *m = nullptr;
    {
        std::lock_guard<std::mutex> lk(g_mu);
        auto it = g_mailboxes.find(id);
        if (it == g_mailboxes.end()) return fail(PSX_EINVAL, "unknown mailbox id");
        m = it->second;
        g_mailboxes.erase(it);
    }
    cudaSetDevice(m->device);
    cudaDeviceSynchronize();
    cudaFree(m->counter);
    delete m;
    return PSX_OK;
}

int psx_shard_register_mailbox(uint64_t shard_id, int slot, const void *mailbox_handle)
{
    Shard *s = find(g_shards, shard_id);
    if (!s) return fail(PSX_EINVAL, "unknown shard id");
    if (slot < 0 || slot >= PSX_MAX_SLOTS) return fail(PSX_EINVAL, "slot %d out of range", slot);
    HandleBlob b;
    int rc = check_blob(mailbox_handle, KIND_MAILBOX, &b);
    if (rc) return rc;
    if (s->mailbox[slot]) {
        close_mapped(s->mailbox_map[slot]);
        s->mailbox[slot] = nullptr;
    }
    rc = open_blob(b, s->device, &s->mailbox_map[slot]);
    if (rc) return rc;
    s->mailbox[slot] = (unsigned int *)s->mailbox_map[slot].base;
    return PSX_OK;
}

int psx_wait_mailbox(uint64_t id, uint32_t target, void *stream)
{
    Mailbox *m = find(g_mailboxes, id);
    if (!m) return fail(PSX_EINVAL, "unknown mailbox id");
    PSX_DEVICE(m->device);
    return stream_wait_geq(stream, m->counter, target);
}

int refuse_in_process_wait(Client *c);

int psx_wait_applied(uint64_t client_id, uint32_t seq, void *stream)
{
    Client *c = find(g_clients, client_id);
    if (!c) return fail(PSX_EINVAL, "unknown client id");
    int rc = refuse_in_process_wait(c);
    if (rc) return rc;
    PSX_DEVICE(c->device);
    return stream_wait_geq(stream, &c->block->applied, seq);
}

// ------------------------------------------------ request-free serving ABI --
int psx_serve_start(uint64_t shard_id, int mode, int replicas_to_aggregate, int idle_sleep_us)
{
    Shard *s = find(g_shards, shard_id);
    if (!s) return fail(PSX_EINVAL, "unknown shard id");
    std::lock_guard<std::recursive_mutex> lk(s->serve_mu);
    return serve_start_impl(s, mode, replicas_to_aggregate, idle_sleep_us);
}

int psx_serve_stop(uint64_t shard_id)
{
    Shard *s = find(g_shards, shard_id);
    if (!s) return fail(PSX_EINVAL, "unknown shard id");
    std::lock_guard<std::recursive_mutex> lk(s->serve_mu);
    return serve_stop_impl(s, nullptr, nullptr, nullptr);
}

int psx_serve_stats(uint64_t shard_id, uint64_t *iterations, uint32_t *served, uint32_t *dropped,
                    int64_t *step)
{
    Shard *s = find(g_shards, shard_id);
    if (!s) return fail(PSX_EINVAL, "unknown shard id");
    {
        std::lock_guard<std::recursive_mutex> lk(s->serve_mu);
        if (iterations) *iterations = s->server ? s->server->iterations.load() : 0;
    }
    PSX_DEVICE(s->device);
    // a plain copy on its own stream: does not wait for the queued iterations
    cudaStream_t side = nullptr;
    CU_TRY(cudaStreamCreateWithFlags(&side, cudaStreamNonBlocking));
    ShardHeader h;
    cudaError_t e = cudaMemcpyAsync(&h, s->base, sizeof(h), cudaMemcpyDeviceToHost, side);
    if (e == cudaSuccess) e = cudaStreamSynchronize(side);
    cudaStreamDestroy(side);
    if (e != cudaSuccess) return fail(PSX_ECUDA, "reading serve stats: %s", cudaGetErrorString(e));
    if (served) *served = h.served;
    if (dropped) *dropped = h.dropped;
    if (step) *step = h.step;
    return PSX_OK;
}

int psx_push_stamped(uint64_t client_id, const void *grad_dev, uint64_t off, uint64_t n,
                     int src_dtype, uint32_t seq, uint32_t stamp, void *stream)
{
    Client *c = find(g_clients, client_id);
    if (!c) return fail(PSX_EINVAL, "unknown client id");
    if (c->lay.n_slots == 0) return fail(PSX_ESTATE, "shard was created without gradient slots");
    if (off + n > c->lay.nelem) return fail(PSX_EINVAL, "push range outside shard");
    if (n && !grad_dev) return fail(PSX_EINVAL, "null gradient pointer");
    if (!seq) return fail(PSX_EINVAL, "a stamped push publishes: seq must be non-zero");
    PSX_DEVICE(c->device);
    char *dst = c->my_slot() + off * c->lay.wire_bytes();
    return launch_copy(dst, c->lay.wire, grad_dev, src_dtype, n, c->sm_count, &c->block->ticket,
                       &c->hdr()->slot_seq[c->slot], seq, (cudaStream_t)stream, &c->hdr()->arrivals,
                       &c->hdr()->slot_stamp[c->slot], stamp);
}

// A stream wait on a shard that is SERVED BY THIS SAME PROCESS would be submitted
// before the apply that satisfies it; if the two streams share a hardware channel
// the apply queues up behind the wait for ever (see "request-free serving" above).
// Refuse loudly instead of hanging: in-process clients poll (psx_client_poll).
int refuse_in_process_wait(Client *c)
{
    if (c->shard.ipc) return PSX_OK;              // the shard lives in another process
    std::lock_guard<std::mutex> lk(g_mu);
    for (auto &kv : g_shards)
        if (kv.second->base == c->shard.base && kv.second->server != nullptr)
            return fail(PSX_ESTATE, "this process serves the shard itself: a stream wait on it can "
                                    "deadlock behind the serving stream's hardware channel -- poll "
                                    "with psx_client_poll (workers normally live in their own process)");
    return PSX_OK;
}

int psx_wait_tokens(uint64_t client_id, uint32_t target, void *stream)
{
    Client *c = find(g_clients, client_id);
    if (!c) return fail(PSX_EINVAL, "unknown client id");
    int rc = refuse_in_process_wait(c);
    if (rc) return rc;
    PSX_DEVICE(c->device);
    return stream_wait_geq(stream, &c->block->tokens, target);
}

int psx_client_poll(uint64_t client_id, uint32_t *applied, uint32_t *tokens, int64_t *step,
                    int *in_process)
{
    Client *c = find(g_clients, client_id);
    if (!c) return fail(PSX_EINVAL, "unknown client id");
    if (in_process) *in_process = c->shard.ipc ? 0 : 1;
    PSX_DEVICE(c->device);
    {
        std::lock_guard<std::mutex> lk(g_mu);     // two pollers must not both create it
        if (!c->poll_stream) CU_TRY(cudaStreamCreateWithFlags(&c->poll_stream, cudaStreamNonBlocking));
    }
    ClientBlock b;
    CU_TRY(cudaMemcpyAsync(&b, c->block, sizeof(b), cudaMemcpyDeviceToHost, c->poll_stream));
    CU_TRY(cudaStreamSynchronize(c->poll_stream));
    if (applied) *applied = b.applied;
    if (tokens) *tokens = b.tokens;
    if (step) *step = b.step;
    return PSX_OK;
}

int psx_read_step_async(uint64_t client_id, int64_t *host_pinned, void *stream)
{
    Client *c = find(g_clients, client_id);
    if (!c || !host_pinned) return fail(PSX_EINVAL, "unknown client id or null destination");
    PSX_DEVICE(c->device);
    CU_TRY(cudaMemcpyAsync(host_pinned, &c->block->step, sizeof(int64_t), cudaMemcpyDeviceToHost,
                           (cudaStream_t)stream));
    return PSX_OK;
}

// ------------------------------------------------ index-list (sparse) rows --
int psx_push_rows(uint64_t client_id, const int64_t *idx_dev, const void *rows_dev, uint64_t k,
                  uint64_t row_len, int src_dtype, uint32_t seq, void *stream)
{
    Client *c = find(g_clients, client_id);
    if (!c) return fail(PSX_EINVAL, "unknown client id");
    if (c->lay.n_slots == 0) return fail(PSX_ESTATE, "shard was created without gradient slots");
    if (!seq) return fail(PSX_EINVAL, "a row push publishes: seq must be non-zero");
    if (row_len == 0 || c->lay.nelem % row_len) return fail(PSX_EINVAL, "row_len %llu does not divide the shard's %llu elements", (unsigned long long)row_len, (unsigned long long)c->lay.nelem);
    if (k && (!idx_dev || !rows_dev)) return fail(PSX_EINVAL, "null index / row pointer");
    const size_t need = rows_data_off(k) + k * row_len * c->lay.wire_bytes();
    if (need > c->lay.nelem_pad * c->lay.wire_bytes())
        return fail(PSX_EINVAL, "%llu rows of %llu do not fit the landing slot (%zu > %zu bytes)", (unsigned long long)k, (unsigned long long)row_len, need, (size_t)(c->lay.nelem_pad * c->lay.wire_bytes()));
    PSX_DEVICE(c->device);
    const int grid = grid_for(k * row_len ? k * row_len : 1, kCopyThreads, c->sm_count, 8);
    unsigned int *flag = &c->hdr()->slot_seq[c->slot];
    unsigned int *arr = &c->hdr()->arrivals;
    cudaStream_t st = (cudaStream_t)stream;
#define PSX_PR(S, D) k_push_rows<S, D><<<grid, kCopyThreads, 0, st>>>(c->my_slot(), (const long long *)idx_dev, (const S *)rows_dev, (size_t)k, (size_t)row_len, &c->block->ticket, flag, arr, seq)
    const int dt = c->lay.wire;
    if (src_dtype == PSX_F32 && dt == PSX_F32) PSX_PR(float, float);
    else if (src_dtype == PSX_F32 && dt == PSX_BF16) PSX_PR(float, __nv_bfloat16);
    else if (src_dtype == PSX_BF16 && dt == PSX_F32) PSX_PR(__nv_bfloat16, float);
    else if (src_dtype == PSX_BF16 && dt == PSX_BF16) PSX_PR(__nv_bfloat16, __nv_bfloat16);
    else return fail(PSX_EINVAL, "unknown dtype %d", src_dtype);
#undef PSX_PR
    LAUNCH_CHECK();
    return PSX_OK;
}

int psx_apply_rows(uint64_t id, int mode, int first_slot, int count, uint64_t row_len,
                   uint32_t wait_seq, void *stream)
{
    Shard *s = find(g_shards, id);
    if (!s) return fail(PSX_EINVAL, "unknown shard id");
    int rc = check_range(first_slot, count, s->lay.n_slots);
    if (rc) return rc;
    if (row_len == 0 || s->lay.nelem % row_len) return fail(PSX_EINVAL, "row_len does not divide the shard");
    if (mode != PSX_MODE_SUM && mode != PSX_MODE_SYNC_MEAN)
        return fail(PSX_EINVAL, "row applies aggregate (SUM / SYNC_MEAN); apply slots one by one for async");
    PSX_DEVICE(s->device);
    rc = wait_slots(s, first_slot, count, wait_seq, stream);
    if (rc) return rc;
    PeerSet peers;
    memset(&peers, 0, sizeof(peers));
    fill_mirrors(s, &peers);
    const size_t stride = (size_t)s->lay.nelem_pad * s->lay.wire_bytes();
    const size_t n_rows = s->lay.nelem / row_len;
    const int grid = s->sm_count * 4;
    cudaStream_t st = (cudaStream_t)stream;
#define PSX_AR(O, M, W) k_apply_rows<O, M, W><<<grid, 256, 0, st>>>(s->hdr(), s->var(), s->m(), s->v(), s->slot(0), stride, first_slot, count, (size_t)row_len, n_rows, peers)
#define PSX_AR2(O, M) do { if (s->lay.wire == PSX_F32) PSX_AR(O, M, float); else PSX_AR(O, M, __nv_bfloat16); } while (0)
    const int opt = s->lay.opt;
#define PSX_AR3(O) do { if (mode == PSX_MODE_SUM) PSX_AR2(O, PSX_MODE_SUM); else PSX_AR2(O, PSX_MODE_SYNC_MEAN); } while (0)
    if (opt == PSX_OPT_SGD) PSX_AR3(PSX_OPT_SGD);
    else if (opt == PSX_OPT_ADAM) PSX_AR3(PSX_OPT_ADAM);
    else if (opt == PSX_OPT_MOMENTUM) PSX_AR3(PSX_OPT_MOMENTUM);
    else if (opt == PSX_OPT_ADAGRAD) PSX_AR3(PSX_OPT_ADAGRAD);
    else if (opt == PSX_OPT_RMSPROP) PSX_AR3(PSX_OPT_RMSPROP);
    else return fail(PSX_EINVAL, "unknown optimizer %d", opt);
#undef PSX_AR3
#undef PSX_AR2
#undef PSX_AR
    LAUNCH_CHECK();
    return PSX_OK;
}

// ----------------------------------------------------------- tensor lists ---
int psx_list_create(uint64_t client_id, const void *const *dev_ptrs, const uint64_t *offs,
                    const uint64_t *n, int count, uint64_t *out_list_id)
{
    Client *c = find(g_clients, client_id);
    if (!c) return fail(PSX_EINVAL, "unknown client id");
    if (!dev_ptrs || !offs || !n || !out_list_id || count < 1) return fail(PSX_EINVAL, "bad list arguments");
    if (c->lay.wire != PSX_F32) return fail(PSX_ESTATE, "tensor lists need an f32 wire format");
    std::vector<ListChunk> chunks;
    for (int i = 0; i < count; ++i) {
        if (offs[i] + n[i] > c->lay.nelem)
            return fail(PSX_EINVAL, "tensor %d: [%llu,+%llu) outside shard of %llu", i,
                        (unsigned long long)offs[i], (unsigned long long)n[i],
                        (unsigned long long)c->lay.nelem);
        if (n[i] == 0) continue;
        if (!dev_ptrs[i]) return fail(PSX_EINVAL, "tensor %d: null pointer", i);
        char *t = (char *)dev_ptrs[i];
        uint64_t soff = offs[i] * 4, bytes = n[i] * 4;
        const bool aligned = ((uintptr_t)t % 16 == 0) && (soff % 16 == 0);
        uint64_t body = aligned ? bytes / 16 * 16 : 0;
        for (uint64_t b = 0; b < body; b += kListChunkBytes) {
            ListChunk ch;
            ch.tensor = t + b;
            ch.shard_off = soff + b;
            ch.bytes = (uint32_t)((body - b) < kListChunkBytes ? (body - b) : kListChunkBytes);
            ch.plain = 0;
            chunks.push_back(ch);
        }
        for (uint64_t b = body; b < bytes; b += kListChunkBytes) {   // ragged tail / unaligned tensor
            ListChunk ch;
            ch.tensor = t + b;
            ch.shard_off = soff + b;
            ch.bytes = (uint32_t)((bytes - b) < kListChunkBytes ? (bytes - b) : kListChunkBytes);
            ch.plain = 1;
            chunks.push_back(ch);
        }
    }
    if (chunks.empty()) return fail(PSX_EINVAL, "empty tensor list");
    PSX_DEVICE(c->device);
    TensorList *l = new TensorList();
    l->client_id = client_id;
    l->device = c->device;
    l->n_chunks = (int)chunks.size();
    l->sm_count = c->sm_count;
    cudaError_t e = cudaMalloc((void **)&l->d_chunks, chunks.size() * sizeof(ListChunk));
    if (e == cudaSuccess)
        e = cudaMemcpy(l->d_chunks, chunks.data(), chunks.size() * sizeof(ListChunk), cudaMemcpyHostToDevice);
    if (e == cudaSuccess)
        e = cudaFuncSetAttribute(k_list_tma, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 kListStages * kListChunkBytes);
    if (e != cudaSuccess) {
        cudaFree(l->d_chunks);
        delete l;
        return fail(PSX_ECUDA, "creating tensor list: %s", cudaGetErrorString(e));
    }
    uint64_t id = g_next_id.fetch_add(1);
    {
        std::lock_guard<std::mutex> lk(g_mu);
        g_lists[id] = l;
    }
    *out_list_id = id;
    return PSX_OK;
}

int psx_list_destroy(uint64_t list_id)
{
    TensorList *l = nullptr;
    {
        std::lock_guard<std::mutex> lk(g_mu);
        auto it = g_lists.find(list_id);
        if (it == g_lists.end()) return fail(PSX_EINVAL, "unknown list id");
        l = it->second;
        g_lists.erase(it);
    }
    cudaSetDevice(l->device);
    cudaDeviceSynchronize();
    cudaFree(l->d_chunks);
    delete l;
    return PSX_OK;
}

static int launch_list(TensorList *l, Client *c, int to_shard, int use_tma, unsigned int *flag,
                       uint32_t seq, cudaStream_t st)
{
    unsigned int *arrivals = flag ? &c->hdr()->arrivals : nullptr;
    char *base = to_shard ? c->my_slot() : (char *)c->var();
    unsigned int *ticket = &c->block->ticket;
    if (use_tma) {
        // 64 KiB of shared memory per CTA -> 3 CTAs per SM
        int grid = l->n_chunks < l->sm_count * 3 ? l->n_chunks : l->sm_count * 3;
        k_list_tma<<<grid, kListThreads, kListStages * kListChunkBytes, st>>>(
            l->d_chunks, l->n_chunks, base, to_shard, ticket, flag, arrivals, seq);
    } else {
        int grid = l->n_chunks < l->sm_count * 16 ? l->n_chunks : l->sm_count * 16;
        k_list_ldst<<<grid, kListThreads, 0, st>>>(l->d_chunks, l->n_chunks, base, to_shard, ticket,
                                                    flag, arrivals, seq);
    }
    LAUNCH_CHECK();
    return PSX_OK;
}

int psx_push_list(uint64_t list_id, uint32_t seq, int use_tma, void *stream)
{
    TensorList *l = find(g_lists, list_id);
    if (!l) return fail(PSX_EINVAL, "unknown list id");
    Client *c = find(g_clients, l->client_id);
    if (!c) return fail(PSX_ESTATE, "the list's client was closed");
    if (c->lay.n_slots == 0) return fail(PSX_ESTATE, "shard was created without gradient slots");
    PSX_DEVICE(c->device);
    return launch_list(l, c, 1, use_tma, seq ? &c->hdr()->slot_seq[c->slot] : nullptr, seq,
                       (cudaStream_t)stream);
}

int psx_pull_list(uint64_t list_id, uint32_t wait_seq, int use_tma, void *stream)
{
    TensorList *l = find(g_lists, list_id);
    if (!l) return fail(PSX_EINVAL, "unknown list id");
    Client *c = find(g_clients, l->client_id);
    if (!c) return fail(PSX_ESTATE, "the list's client was closed");
    PSX_DEVICE(c->device);
    if (wait_seq) {
        int rc = stream_wait_geq(stream, &c->block->applied, wait_seq);
        if (rc) return rc;
    }
    return launch_list(l, c, 0, use_tma, nullptr, 0, (cudaStream_t)stream);
}

// ----------------------------------------------------------- fused round ----
int psx_buffer_create(int device, uint64_t nbytes, uint64_t *out_id, void **out_dev_ptr)
{
    if (!out_id || !out_dev_ptr || nbytes == 0) return fail(PSX_EINVAL, "bad buffer arguments");
    PSX_DEVICE(device);
    void *p = nullptr;
    cudaError_t e = cudaMalloc(&p, nbytes);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(e == cudaErrorMemoryAllocation ? PSX_ENOMEM : PSX_ECUDA, "cudaMalloc(%llu): %s",
                    (unsigned long long)nbytes, cudaGetErrorString(e));
    }
    CU_TRY(cudaMemset(p, 0, nbytes));
    Buffer *b = new Buffer();
    b->device = device;
    b->nbytes = nbytes;
    b->base = (char *)p;
    uint64_t id = g_next_id.fetch_add(1);
    {
        std::lock_guard<std::mutex> lk(g_mu);
        g_buffers[id] = b;
    }
    *out_id = id;
    *out_dev_ptr = p;
    return PSX_OK;
}

int psx_buffer_export(uint64_t id, void *out_handle)
{
    Buffer *bf = find(g_buffers, id);
    if (!bf || !out_handle) return fail(PSX_EINVAL, "unknown buffer id or null handle");
    HandleBlob b;
    memset(&b, 0, sizeof(b));
    b.magic = kMagic;
    b.abi = PSX_ABI_VERSION;
    b.kind = KIND_BUFFER;
    b.device = bf->device;
    b.pid = (uint64_t)getpid();
    b.local_id = id;
    b.nelem = bf->nbytes;
    PSX_DEVICE(bf->device);
    CU_TRY(cudaIpcGetMemHandle(&b.ipc, bf->base));
    memcpy(out_handle, &b, sizeof(b));
    return PSX_OK;
}

int psx_buffer_destroy(uint64_t id)
{
    Buffer *b = nullptr;
    {
        std::lock_guard<std::mutex> lk(g_mu);
        auto it = g_buffers.find(id);
        if (it == g_buffers.end()) return fail(PSX_EINVAL, "unknown buffer id");
        b = it->second;
        g_buffers.erase(it);
    }
    cudaSetDevice(b->device);
    cudaDeviceSynchronize();
    cudaFree(b->base);
    delete b;
    return PSX_OK;
}

int psx_round_bind(uint64_t shard_id, int slot, const void *grad_buf_handle,
                   const void *param_buf_handle, uint64_t elem_off)
{
    Shard *s = find(g_shards, shard_id);
    if (!s) return fail(PSX_EINVAL, "unknown shard id");
    if (slot < 0 || slot >= PSX_MAX_SLOTS) return fail(PSX_EINVAL, "slot %d out of range", slot);
    if (elem_off % 4) return fail(PSX_EINVAL, "elem_off must be a multiple of 4 (16-byte vectors)");
    HandleBlob g, p;
    int rc = check_blob(grad_buf_handle, KIND_BUFFER, &g);
    if (rc) return rc;
    rc = check_blob(param_buf_handle, KIND_BUFFER, &p);
    if (rc) return rc;
    // the kernel touches nelem_pad elements (of the shard's wire dtype) of every bound buffer
    const uint64_t need = (elem_off + s->lay.nelem_pad) * s->lay.wire_bytes();
    if (g.nelem < need || p.nelem < need)
        return fail(PSX_EINVAL, "bound buffers must hold %llu bytes (elem_off + padded shard), have %llu/%llu",
                    (unsigned long long)need, (unsigned long long)g.nelem, (unsigned long long)p.nelem);
    Bound &b = s->bound[slot];
    if (b.valid) {
        close_mapped(b.grad);
        close_mapped(b.param);
        b.valid = false;
    }
    rc = open_blob(g, s->device, &b.grad);
    if (rc) return rc;
    rc = open_blob(p, s->device, &b.param);
    if (rc) {
        close_mapped(b.grad);
        return rc;
    }
    b.elem_off = elem_off;
    b.valid = true;
    return PSX_OK;
}

static int round_impl(uint64_t shard_id, int mode, int first_slot, int count, uint32_t wait_seq,
                      int counted, void *stream)
{
    Shard *s = find(g_shards, shard_id);
    if (!s) return fail(PSX_EINVAL, "unknown shard id");
    int rc = check_range(first_slot, count, PSX_MAX_SLOTS);
    if (rc) return rc;
    PeerSet peers;
    memset(&peers, 0, sizeof(peers));
    fill_mirrors(s, &peers);
    const size_t wb = s->lay.wire_bytes();
    const bool nvls = s->mc_grad != nullptr;
    if (nvls) {
        // the switch sums ALL members' gradient copies: the round is over every worker
        if (first_slot != 0 || count != s->mc_members)
            return fail(PSX_EINVAL, "an NVLS round covers all %d workers (got slots [%d,%d))",
                        s->mc_members, first_slot, first_slot + count);
        if (mode == PSX_MODE_ASYNC_ORDERED)
            return fail(PSX_ESTATE, "the NVLS round reduces in the switch: SUM / SYNC_MEAN only");
        peers.mc_param = s->mc_param;
    } else {
        for (int k = 0; k < count; ++k) {
            const Bound &b = s->bound[first_slot + k];
            if (!b.valid) return fail(PSX_ESTATE, "slot %d has no bound buffers (psx_round_bind)", first_slot + k);
            peers.grad[first_slot + k] = b.grad.base + b.elem_off * wb;
        }
        for (int c = 0; c < PSX_MAX_SLOTS; ++c)  // every bound worker receives the new parameters
            if (s->bound[c].valid)
                peers.param[peers.n_param++] = s->bound[c].param.base + s->bound[c].elem_off * wb;
    }
    PSX_DEVICE(s->device);
    if (counted) {
        rc = stream_wait_geq(stream, &s->hdr()->arrivals, (uint32_t)count);
    } else {
        // slot flags exist for all PSX_MAX_SLOTS slots, whether or not the shard has
        // landing slots (psx_round needs none)
        rc = wait_slots(s, first_slot, count, wait_seq, stream);
    }
    if (rc) return rc;
    const ApplyRange r{0, (size_t)s->lay.nelem_pad, 1, counted ? (unsigned int)count : 0u, count};
    if (nvls) return launch_round_mc(s, mode, peers, (cudaStream_t)stream, r);
    if (s->lay.wire == PSX_F32) {
        PeerSrc<float> src{peers, first_slot};
        return launch_apply<true>(s, mode, src, count, peers, (cudaStream_t)stream, r);
    }
    PeerSrc<__nv_bfloat16> src{peers, first_slot};
    return launch_apply<true>(s, mode, src, count, peers, (cudaStream_t)stream, r);
}

int psx_round(uint64_t shard_id, int mode, int first_slot, int count, uint32_t wait_seq, void *stream)
{
    return round_impl(shard_id, mode, first_slot, count, wait_seq, 0, stream);
}

int psx_round_counted(uint64_t shard_id, int mode, int first_slot, int count, void *stream)
{
    return round_impl(shard_id, mode, first_slot, count, 0, 1, stream);
}

int psx_batch(const psx_op *ops, int n_ops, int *failed_index)
{
    if (!ops || n_ops < 0) return fail(PSX_EINVAL, "bad batch");
    for (int i = 0; i < n_ops; ++i) {
        const psx_op &o = ops[i];
        int rc;
        switch (o.op) {
        case PSX_OP_PUSH: rc = psx_push(o.id, o.ptr, o.off, o.n, o.a, o.seq, o.stream); break;
        case PSX_OP_PULL: rc = psx_pull(o.id, o.ptr, o.off, o.n, o.a, o.seq, o.stream); break;
        case PSX_OP_APPLY: rc = psx_apply(o.id, o.a, o.b, o.c, o.seq, o.stream); break;
        case PSX_OP_ROUND: rc = psx_round(o.id, o.a, o.b, o.c, o.seq, o.stream); break;
        case PSX_OP_SIGNAL: rc = psx_signal(o.id, o.seq, o.stream); break;
        case PSX_OP_WAIT_APPLIED: rc = psx_wait_applied(o.id, o.seq, o.stream); break;
        case PSX_OP_WAIT_SLOTS: rc = psx_wait_slots(o.id, o.b, o.c, o.seq, o.stream); break;
        case PSX_OP_SIGNAL_MANY: rc = psx_signal_many((const uint64_t *)o.ptr, (int)o.n, o.seq, o.stream); break;
        case PSX_OP_WAIT_ARRIVALS: rc = psx_wait_arrivals(o.id, o.seq * (uint32_t)o.c, o.stream); break;
        case PSX_OP_WAIT_MAILBOX: rc = psx_wait_mailbox(o.id, o.seq * (uint32_t)o.c, o.stream); break;
        case PSX_OP_ROUND_COUNTED: rc = psx_round_counted(o.id, o.a, o.b, o.c, o.stream); break;
        case PSX_OP_APPLY_COUNTED: rc = psx_apply_counted(o.id, o.a, o.b, o.c, o.stream); break;
        case PSX_OP_SIGNAL_COUNTED:
            rc = psx_signal_counted((const uint64_t *)o.ptr, (int)o.n, o.seq, o.id, (uint32_t)o.c, o.stream);
            break;
        case PSX_OP_MAILBOX_WAIT: rc = psx_wait_mailbox(o.id, (uint32_t)o.c, o.stream); break;
        case PSX_OP_MAILBOX_CONSUME: rc = psx_mailbox_consume(o.id, (uint32_t)o.c, o.stream); break;
        default: rc = fail(PSX_EINVAL, "batch op %d: unknown opcode %d", i, o.op);
        }
        if (rc) {
            if (failed_index) *failed_index = i;
            return rc;
        }
    }
    return PSX_OK;
}

int psx_copy(int device, void *dst, const void *src, uint64_t nbytes, void *stream)
{
    if (nbytes % 4) return fail(PSX_EINVAL, "nbytes must be a multiple of 4");
    PSX_DEVICE(device);
    return launch_copy(dst, PSX_F32, src, PSX_F32, nbytes / 4, sm_count_of(device), nullptr, nullptr, 0,
                       (cudaStream_t)stream);
}

}  // extern "C"

#include "psx_nvls.cuh"
