// psx_kernels.cuh -- sm_100a device code of the parameter-server data plane.
//
// Every kernel here is HBM- or NVLink-bound elementwise work (SURVEY.md 8d:
// no dense contraction on the push/apply/pull path, so no tensor cores):
//   * 128-bit vector loads/stores, fully coalesced, streaming cache hints
//   * grids sized to the resident capacity of the 148 SMs, grid-stride loops
//   * gradients reduced in registers in a FIXED slot order
//   * arithmetic spelled with __f*_rn intrinsics: one IEEE-754 rounding per
//     operation, never contracted to FMA, so results are bit-identical to the
//     CPU restatements of TF 0.12's ApplyGradientDescent / ApplyAdam /
//     ApplyMomentum / ApplyAdagrad / ApplyRMSProp
//   * completion published with a last-CTA ticket + fence.sys + system-scope flag store so the
//     consumer (another GPU / another process) can wait with a stream memop
//     instead of a spinning kernel.
#pragma once

#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#include "psx.h"

namespace psx {

// ---------------------------------------------------------------- layout ----
// First 4 KiB of every shard allocation.  Lives in the PS GPU's HBM; workers
// map it (CUDA IPC) to publish their slot flags.
struct ShardHeader {
    uint32_t magic;
    uint32_t abi;
    float lr, b1, b2, eps;            // hyper-parameters (mnist_replica.py:147)
    float b1p, b2p;                   // stored beta powers (AdamOptimizer._finish)
    long long step;                   // global_step (mnist.py:46, mnist_replica.py:121)
    unsigned int ticket;              // last-CTA counter of the apply kernels
    unsigned int apply_seq;           // completed apply rounds
    unsigned int slot_seq[PSX_MAX_SLOTS];  // round number last pushed into slot s
    unsigned int arrivals;            // +1 per completed push / signal (any slot): lets the
                                      // PS wait for "all W workers of round r" with ONE memop
    // ---- request-free serving (psx_serve_start): the PS consumes pushes as they ARRIVE
    unsigned int reserved0;
    unsigned int pick_n;              // slots the current iteration's apply consumes ...
    unsigned int pick[PSX_MAX_SLOTS]; // ... in this order (arrival order between picks)
    unsigned int pick_seq[PSX_MAX_SLOTS];   // push sequence number consumed per picked slot
    unsigned int slot_seen[PSX_MAX_SLOTS];  // last push of slot s the picker has looked at
    unsigned int slot_stamp[PSX_MAX_SLOTS]; // global_step the pushed gradient was computed at
                                            // (SyncReplicas' local_step, mnist_replica.py:148-154)
    unsigned int pending[PSX_MAX_SLOTS];    // sync mode: fresh gradient waiting for aggregation
    unsigned int arrival_rank[PSX_MAX_SLOTS];
    unsigned int arrival_ctr;
    unsigned int dropped;             // gradients discarded as stale (sync mode)
    unsigned int served;              // pushes consumed by applies
    unsigned long long client_block[PSX_MAX_SLOTS];  // PS-side address of each registered worker's
                                      // ClientBlock (0 = none): read by the served epilogue at RUN
                                      // time, so a worker may register while iterations are queued
};
static_assert(sizeof(ShardHeader) <= 4096, "header must fit its page");

// Worker-local block (in the WORKER GPU's HBM): ticket for its push kernels and
// the mirror of the shard's apply_seq the PS writes remotely.
struct ClientBlock {
    unsigned int ticket;
    unsigned int applied;             // mirror of ShardHeader::apply_seq; in served mode: the
                                      // sequence number of THIS worker's last consumed push
    long long step;                   // served mode: global_step after that apply (what
                                      // sess.run([train_step, global_step]) returns)
    unsigned int tokens;              // served sync mode: one token per aggregated apply
    unsigned int pad[59];
};
static_assert(sizeof(ClientBlock) == 256, "client block is 256 bytes");

struct PeerSet {                      // by-value kernel argument (PS address space)
    const void *grad[PSX_MAX_SLOTS];  // bound worker gradient buffers (psx_round), wire dtype
    void *param[PSX_MAX_SLOTS];       // bound worker parameter buffers, compact, wire dtype
    unsigned int *mirror[PSX_MAX_SLOTS];  // ClientBlock::applied of each client, compact
    unsigned int *mailbox[PSX_MAX_SLOTS]; // per-worker completion counters, compact
    float *mc_param;                      // NVLS: multicast address of every worker's parameter
                                          // buffer (one multimem.st reaches all of them)
    int n_param;
    int n_mirror;
    int n_mailbox;
};

// ------------------------------------------------------------ primitives ----
// Flag publication = ONE system-scope fence (__threadfence_system, issued by the
// caller right before) followed by relaxed system-scope stores / reductions: the
// fence orders everything before it ahead of all of them, so a kernel that
// publishes to 8 mirrors + 8 mailboxes pays one MEMBAR.SYS, not seventeen
// (a .release store carries its own fence; ~2.5 us each -- profiles/r07).
__device__ __forceinline__ void publish_store(unsigned int *p, unsigned int v)
{
    asm volatile("st.relaxed.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ void publish_add(unsigned int *p, unsigned int v)
{
    asm volatile("red.relaxed.sys.global.add.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// the arrival counter is bumped AFTER the slot flag it announces (release: the flag
// store above is ordered before it), so a picker woken by the counter finds the flag
__device__ __forceinline__ void publish_add_release(unsigned int *p, unsigned int v)
{
    asm volatile("red.release.sys.global.add.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned int ld_sys(const unsigned int *p)
{
    unsigned int v;
    asm volatile("ld.relaxed.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

// streaming (read-once) 128-bit load; works on local and peer-mapped addresses
__device__ __forceinline__ float4 ld_stream(const float4 *p)
{
    float4 r;
    asm volatile("ld.global.cs.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
                 : "l"(p));
    return r;
}
__device__ __forceinline__ void st_stream(float4 *p, const float4 &v)
{
    asm volatile("st.global.cs.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y),
                 "f"(v.z), "f"(v.w)
                 : "memory");
}
__device__ __forceinline__ uint2 ld_stream(const uint2 *p)
{
    uint2 r;
    asm volatile("ld.global.cs.v2.u32 {%0,%1}, [%2];" : "=r"(r.x), "=r"(r.y) : "l"(p));
    return r;
}
__device__ __forceinline__ void st_stream(uint2 *p, const uint2 &v)
{
    asm volatile("st.global.cs.v2.u32 [%0], {%1,%2};" ::"l"(p), "r"(v.x), "r"(v.y) : "memory");
}

// 4-element vectors of the two wire types
template <typename T> struct Vec4;
template <> struct Vec4<float> {
    static __device__ __forceinline__ float4 load(const float *p) { return ld_stream((const float4 *)p); }
    static __device__ __forceinline__ void store(float *p, const float4 &v) { st_stream((float4 *)p, v); }
};
template <> struct Vec4<__nv_bfloat16> {
    static __device__ __forceinline__ float4 load(const __nv_bfloat16 *p)
    {
        uint2 u = ld_stream((const uint2 *)p);
        float4 r;  // bf16 -> f32 is exact: place the 16 bits in the high half
        r.x = __uint_as_float(u.x << 16);
        r.y = __uint_as_float(u.x & 0xffff0000u);
        r.z = __uint_as_float(u.y << 16);
        r.w = __uint_as_float(u.y & 0xffff0000u);
        return r;
    }
    static __device__ __forceinline__ void store(__nv_bfloat16 *p, const float4 &v)
    {
        // round-to-nearest-even, identical to psx_oracle_f32_to_bf16
        __nv_bfloat162 lo = __floats2bfloat162_rn(v.x, v.y);
        __nv_bfloat162 hi = __floats2bfloat162_rn(v.z, v.w);
        uint2 u;
        u.x = *reinterpret_cast<unsigned int *>(&lo);
        u.y = *reinterpret_cast<unsigned int *>(&hi);
        st_stream((uint2 *)p, u);
    }
};

template <typename T> __device__ __forceinline__ float to_f32(T v);
template <> __device__ __forceinline__ float to_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ float to_f32<__nv_bfloat16>(__nv_bfloat16 v) { return __bfloat162float(v); }
template <typename T> __device__ __forceinline__ T from_f32(float v);
template <> __device__ __forceinline__ float from_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ __nv_bfloat16 from_f32<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }

// Grid-wide completion: the last CTA to arrive publishes `seq` in *flag (which
// may live in another GPU's HBM).  bar.sync, then thread 0: fence at GPU scope
// (orders every write of this CTA before its ticket, cumulatively), ticket; the
// CTA that draws the last ticket has thereby observed all the others, issues ONE
// system-scope fence and stores the flag(s).  (A MEMBAR.SYS costs ~3 us;
// paying it once per kernel instead of once per CTA is what keeps 300 KB
// MNIST-sized rounds in the 10 us range -- profiles/r01.)
template <bool SYS_FENCE = false>
__device__ __forceinline__ bool last_cta(unsigned int *ticket)
{
    __shared__ bool s_last;
    __syncthreads();
    if (threadIdx.x == 0) {
        // SYS_FENCE: the CTA's own writes went through the NVSwitch multicast path
        // (multimem.st); order them at system scope here instead of relying on the
        // last CTA's fence to cover other SMs' in-switch replications
        if (SYS_FENCE) __threadfence_system();
        else __threadfence();
        unsigned int t = atomicAdd(ticket, 1u);
        s_last = (t == gridDim.x - 1);
    }
    __syncthreads();
    return s_last;
}

// ------------------------------------------------------------ push / pull ----
// dst[0..n) = cast(src[0..n)).  One kernel serves PUSH (dst = slot in the PS
// shard, possibly across NVLink) and PULL (src = var in the PS shard).  Tiles
// of 256 threads x UNROLL vectors; all loads of a tile are issued before its
// stores (memory-level parallelism for the ~2-3.7 us NVLink round trip).
constexpr int kCopyThreads = 256;
constexpr int kCopyUnroll = 4;

template <typename SRC, typename DST>
__global__ void __launch_bounds__(kCopyThreads)
k_copy(DST *__restrict__ dst, const SRC *__restrict__ src, size_t n, int vec_ok,
       unsigned int *ticket, unsigned int *flag, unsigned int *arrivals, unsigned int seq,
       unsigned int *stamp_word = nullptr, unsigned int stamp = 0)
{
    if (vec_ok) {
        const size_t n4 = n >> 2;
        const size_t tile = (size_t)kCopyThreads * kCopyUnroll;
        const size_t tiles = (n4 + tile - 1) / tile;
        for (size_t t = blockIdx.x; t < tiles; t += gridDim.x) {
            const size_t base = t * tile + threadIdx.x;
            float4 r[kCopyUnroll];
#pragma unroll
            for (int u = 0; u < kCopyUnroll; ++u) {
                size_t i = base + (size_t)u * kCopyThreads;
                if (i < n4) r[u] = Vec4<SRC>::load(src + 4 * i);
            }
#pragma unroll
            for (int u = 0; u < kCopyUnroll; ++u) {
                size_t i = base + (size_t)u * kCopyThreads;
                if (i < n4) Vec4<DST>::store(dst + 4 * i, r[u]);
            }
        }
        // scalar tail (< 4 elements)
        if (blockIdx.x == 0 && threadIdx.x < (n & 3)) {
            size_t i = (n4 << 2) + threadIdx.x;
            dst[i] = from_f32<DST>(to_f32<SRC>(src[i]));
        }
    } else {  // unaligned sub-range: correct, not fast
        for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n;
             i += (size_t)gridDim.x * blockDim.x)
            dst[i] = from_f32<DST>(to_f32<SRC>(src[i]));
    }
    if (flag != nullptr) {
        if (last_cta(ticket) && threadIdx.x == 0) {
            *ticket = 0;
            if (stamp_word != nullptr) publish_store(stamp_word, stamp);   // ordered by the fence below
            __threadfence_system();
            publish_store(flag, seq);
            if (arrivals != nullptr) publish_add_release(arrivals, 1u);
        }
    }
}

// ------------------------------------------------------- tensor lists (TMA) ----
// A model's parameters are a LIST of tensors (ResNet-50: 161, 107 of them
// <= 2048 elements).  One launch moves the whole list between the worker's
// separate tensors and their places in the flat shard: the host cuts every
// tensor into <= 16 KiB chunks once (psx_list_create); each CTA streams its
// chunks global -> shared -> global with bulk-async (TMA) copies through a
// 4-stage shared-memory ring -- one elected thread drives the copy engine, no
// registers or LSU instructions are spent on the data.
struct ListChunk {
    char *tensor;              // worker-side address of this chunk
    uint64_t shard_off;        // byte offset inside the slot / var region
    uint32_t bytes;            // multiple of 16 for TMA chunks
    uint32_t plain;            // 1: not 16 B aligned -> element loop by the whole CTA
};

constexpr int kListStages = 4;
constexpr uint32_t kListChunkBytes = 16384;
constexpr int kListThreads = 128;

__device__ __forceinline__ uint32_t smem_u32(const void *p)
{
    return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
                 "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity)
{
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t"
        "}" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
__device__ __forceinline__ void tma_load_1d(void *smem_dst, const void *gsrc, uint32_t bytes,
                                            uint64_t *bar)
{
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::
            "r"(smem_u32(smem_dst)),
        "l"(gsrc), "r"(bytes), "r"(smem_u32(bar))
        : "memory");
}
__device__ __forceinline__ void tma_store_1d(void *gdst, const void *smem_src, uint32_t bytes)
{
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst),
                 "r"(smem_u32(smem_src)), "r"(bytes)
                 : "memory");
}

// to_shard = 1: PUSH (tensor -> shard_base + off), 0: PULL (shard_base + off -> tensor)
__global__ void __launch_bounds__(kListThreads)
k_list_tma(const ListChunk *__restrict__ chunks, int n_chunks, char *shard_base, int to_shard,
           unsigned int *ticket, unsigned int *flag, unsigned int *arrivals, unsigned int seq)
{
    extern __shared__ __align__(128) unsigned char ring[];
    __shared__ __align__(8) uint64_t full[kListStages];
    if (threadIdx.x == 0) {
        for (int s = 0; s < kListStages; ++s) mbar_init(&full[s], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    __syncthreads();

    const int mine = (n_chunks - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
    auto chunk_of = [&](int j) { return chunks[(size_t)blockIdx.x + (size_t)j * gridDim.x]; };

    if (threadIdx.x == 0) {
        // Ring stage and mbarrier phase are taken from a RUNNING COUNT of the TMA
        // chunks this CTA has issued / consumed, never from the chunk index j:
        // plain chunks (ragged tails, unaligned tensors) sit in between the TMA
        // chunks of a list and issue no load, so indexing by j would leave a
        // stage's barrier one phase behind (stale data or a hang once a CTA owns
        // more than kListStages chunks).
        constexpr int D = kListStages - 2;            // TMA loads kept in flight
        int next_issue = 0;                           // next chunk index to look at for a load
        int issued = 0, consumed = 0;                 // TMA chunks so far
        auto issue_one = [&]() {                      // issue the next TMA chunk, if any
            while (next_issue < mine) {
                const ListChunk c = chunk_of(next_issue++);
                if (c.plain) continue;
                const int s = issued % kListStages;
                const char *src = to_shard ? c.tensor : shard_base + c.shard_off;
                mbar_expect_tx(&full[s], c.bytes);
                tma_load_1d(ring + (size_t)s * kListChunkBytes, src, c.bytes, &full[s]);
                ++issued;
                return;
            }
        };
        for (int k = 0; k < D; ++k) issue_one();
        for (int j = 0; j < mine; ++j) {
            const ListChunk c = chunk_of(j);
            if (c.plain) continue;
            // stage (consumed+D)%S was last read by the store of TMA chunk
            // consumed-2; one bulk group is committed per consumed chunk, so "all
            // but the newest" covers it
            asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
            issue_one();
            const int s = consumed % kListStages;
            mbar_wait(&full[s], (uint32_t)((consumed / kListStages) & 1));
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            char *dst = to_shard ? shard_base + c.shard_off : c.tensor;
            tma_store_1d(dst, ring + (size_t)s * kListChunkBytes, c.bytes);
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            ++consumed;
        }
        asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");   // stores performed
        asm volatile("fence.proxy.async;" ::: "memory");
    }
    // ragged / unaligned tensors: plain element loop by the whole CTA
    for (int j = 0; j < mine; ++j) {
        const ListChunk c = chunk_of(j);
        if (!c.plain) continue;
        const float *src = (const float *)(to_shard ? c.tensor : shard_base + c.shard_off);
        float *dst = (float *)(to_shard ? shard_base + c.shard_off : c.tensor);
        for (uint32_t i = threadIdx.x; i < c.bytes / 4; i += blockDim.x) dst[i] = src[i];
    }
    if (flag != nullptr) {
        if (last_cta(ticket) && threadIdx.x == 0) {
            *ticket = 0;
            __threadfence_system();
            publish_store(flag, seq);
            if (arrivals != nullptr) publish_add(arrivals, 1u);
        }
    }
}

// same table, plain 128-bit loads/stores (the non-TMA baseline of the list path)
__global__ void __launch_bounds__(kListThreads)
k_list_ldst(const ListChunk *__restrict__ chunks, int n_chunks, char *shard_base, int to_shard,
            unsigned int *ticket, unsigned int *flag, unsigned int *arrivals, unsigned int seq)
{
    for (int j = blockIdx.x; j < n_chunks; j += gridDim.x) {
        const ListChunk c = chunks[j];
        const char *src = to_shard ? c.tensor : shard_base + c.shard_off;
        char *dst = to_shard ? shard_base + c.shard_off : c.tensor;
        if (c.plain) {
            for (uint32_t i = threadIdx.x; i < c.bytes / 4; i += blockDim.x)
                ((float *)dst)[i] = ((const float *)src)[i];
        } else {
            const uint32_t n16 = c.bytes / 16;
            for (uint32_t i = threadIdx.x; i < n16; i += 4 * blockDim.x) {
                float4 r[4];
#pragma unroll
                for (int u = 0; u < 4; ++u)
                    if (i + u * blockDim.x < n16) r[u] = ld_stream((const float4 *)src + i + u * blockDim.x);
#pragma unroll
                for (int u = 0; u < 4; ++u)
                    if (i + u * blockDim.x < n16) st_stream((float4 *)dst + i + u * blockDim.x, r[u]);
            }
        }
    }
    if (flag != nullptr) {
        if (last_cta(ticket) && threadIdx.x == 0) {
            *ticket = 0;
            __threadfence_system();
            publish_store(flag, seq);
            if (arrivals != nullptr) publish_add(arrivals, 1u);
        }
    }
}

// one thread: take `n` completions off a worker's mailbox (counted rendez-vous)
// Shard creation: an optimizer state array that does not start at zero.
__global__ void __launch_bounds__(kCopyThreads) k_fill(float4 *__restrict__ dst, float value, size_t n4)
{
    const float4 v = make_float4(value, value, value, value);
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (size_t)gridDim.x * blockDim.x)
        dst[i] = v;
}

__global__ void k_consume(unsigned int *counter, unsigned int n) { atomicSub(counter, n); }

// "my gradients for round seq are in place", to up to kMaxSignal shards in ONE
// launch: thread i publishes slot flag i and bumps that shard's arrival counter
constexpr int kMaxSignal = 64;
struct SignalSet {
    unsigned int *flag[kMaxSignal];
    unsigned int *arrivals[kMaxSignal];
    int n;
    unsigned int *mailbox;      // optional: this worker's mailbox ...
    unsigned int consume;       // ... from which last round's completions are taken first
};
__global__ void k_signal(SignalSet set, unsigned int seq)
{
    if (set.mailbox != nullptr && threadIdx.x == 0) atomicSub(set.mailbox, set.consume);
    if ((int)threadIdx.x < set.n) {
        __threadfence_system();
        publish_store(set.flag[threadIdx.x], seq);
        publish_add(set.arrivals[threadIdx.x], 1u);
    }
}

// --------------------------------------------------------------- optimizer ---
// What each optimizer keeps beside `var`: the number of f32 state arrays (the
// shard's m, v regions) and whether it carries beta powers advanced once per apply.
template <int OPT> struct OptTraits;
template <> struct OptTraits<PSX_OPT_SGD> { static constexpr int kState = 0; static constexpr bool kPowers = false; };
template <> struct OptTraits<PSX_OPT_ADAM> { static constexpr int kState = 2; static constexpr bool kPowers = true; };
template <> struct OptTraits<PSX_OPT_MOMENTUM> { static constexpr int kState = 1; static constexpr bool kPowers = false; };
template <> struct OptTraits<PSX_OPT_ADAGRAD> { static constexpr int kState = 1; static constexpr bool kPowers = false; };
template <> struct OptTraits<PSX_OPT_RMSPROP> { static constexpr int kState = 2; static constexpr bool kPowers = false; };

// TF 0.12 ApplyGradientDescent: var -= grad * lr           (mnist.py:55)
__device__ __forceinline__ float sgd1(float var, float g, float lr)
{
    return __fsub_rn(var, __fmul_rn(g, lr));
}

// TF 0.12 ApplyAdam (mnist_replica.py:147); eps outside the bias correction
__device__ __forceinline__ void adam1(float &var, float &m, float &v, float g, float alpha,
                                      float omb1, float omb2, float eps)
{
    m = __fadd_rn(m, __fmul_rn(__fsub_rn(g, m), omb1));
    v = __fadd_rn(v, __fmul_rn(__fsub_rn(__fmul_rn(g, g), v), omb2));
    float num = __fmul_rn(m, alpha);
    float den = __fadd_rn(__fsqrt_rn(v), eps);
    var = __fsub_rn(var, __fdiv_rn(num, den));
}

// TF 0.12 ApplyMomentum (use_nesterov = false): accum = accum * mu + grad; var -= accum * lr
__device__ __forceinline__ void momentum1(float &var, float &a, float g, float lr, float mu)
{
    a = __fadd_rn(__fmul_rn(a, mu), g);
    var = __fsub_rn(var, __fmul_rn(a, lr));
}

// TF 0.12 ApplyAdagrad: accum += grad^2; var -= grad * lr * rsqrt(accum), with rsqrt
// spelled 1 / sqrt (correctly rounded twice) so the GPU and both CPU restatements agree
__device__ __forceinline__ void adagrad1(float &var, float &a, float g, float lr)
{
    a = __fadd_rn(a, __fmul_rn(g, g));
    var = __fsub_rn(var, __fmul_rn(__fmul_rn(g, lr), __fdiv_rn(1.0f, __fsqrt_rn(a))));
}

// TF 0.12 ApplyRMSProp (not centered): ms += (grad^2 - ms) * (1 - decay);
// mom = mom * mu + grad * lr / sqrt(ms + eps); var -= mom
__device__ __forceinline__ void rmsprop1(float &var, float &ms, float &mom, float g, float lr,
                                         float omdecay, float mu, float eps)
{
    ms = __fadd_rn(ms, __fmul_rn(__fsub_rn(__fmul_rn(g, g), ms), omdecay));
    mom = __fadd_rn(__fmul_rn(mom, mu), __fdiv_rn(__fmul_rn(g, lr), __fsqrt_rn(__fadd_rn(ms, eps))));
    var = __fsub_rn(var, mom);
}

__device__ __forceinline__ float adam_alpha(float lr, float b1p, float b2p)
{
    float s = __fsqrt_rn(__fsub_rn(1.0f, b2p));
    return __fdiv_rn(__fmul_rn(lr, s), __fsub_rn(1.0f, b1p));
}

// One element.  The header's hyper-parameters mean, per optimizer:
//   SGD {lr} | Adam {lr, b1, b2, eps} | Momentum {lr, mu} | Adagrad {lr, init}
//   RMSProp {lr, decay, mu, eps}
// omb1 = 1 - b1 and omb2 = 1 - b2, each rounded once; alpha is Adam's step size.
template <int OPT>
__device__ __forceinline__ void apply1(float &x, float &m, float &v, float g, float lr, float alpha,
                                       float b1, float b2, float omb1, float omb2, float eps)
{
    if (OPT == PSX_OPT_SGD) x = sgd1(x, g, lr);
    else if (OPT == PSX_OPT_ADAM) adam1(x, m, v, g, alpha, omb1, omb2, eps);
    else if (OPT == PSX_OPT_MOMENTUM) momentum1(x, m, g, lr, b1);
    else if (OPT == PSX_OPT_ADAGRAD) adagrad1(x, m, g, lr);
    else rmsprop1(x, m, v, g, lr, omb1, b2, eps);
}

template <int OPT>
__device__ __forceinline__ void apply4(float4 &x, float4 &m, float4 &v, const float4 &g, float lr,
                                       float alpha, float b1, float b2, float omb1, float omb2,
                                       float eps)
{
    apply1<OPT>(x.x, m.x, v.x, g.x, lr, alpha, b1, b2, omb1, omb2, eps);
    apply1<OPT>(x.y, m.y, v.y, g.y, lr, alpha, b1, b2, omb1, omb2, eps);
    apply1<OPT>(x.z, m.z, v.z, g.z, lr, alpha, b1, b2, omb1, omb2, eps);
    apply1<OPT>(x.w, m.w, v.w, g.w, lr, alpha, b1, b2, omb1, omb2, eps);
}

__device__ __forceinline__ float4 add4(const float4 &a, const float4 &b)
{
    return make_float4(__fadd_rn(a.x, b.x), __fadd_rn(a.y, b.y), __fadd_rn(a.z, b.z),
                       __fadd_rn(a.w, b.w));
}
__device__ __forceinline__ float4 div4(const float4 &a, float d)
{
    return make_float4(__fdiv_rn(a.x, d), __fdiv_rn(a.y, d), __fdiv_rn(a.z, d), __fdiv_rn(a.w, d));
}

// Epilogue of every apply / round kernel: the CTA that draws the last ticket
// advances the beta powers and global_step (AdamOptimizer._finish, once per
// apply) and publishes completion to every registered worker.
// finish == 0: a partial (element-range) apply that is not the last of its
// round -- it must not advance the beta powers / global_step / apply_seq.
template <int OPT, bool SYS_FENCE>
__device__ __forceinline__ void finish_apply(ShardHeader *h, const PeerSet &peers, int applies,
                                             int finish, float b1, float b2)
{
    const bool last = last_cta<SYS_FENCE>(&h->ticket);
    if (last && threadIdx.x == 0 && !finish) {
        h->ticket = 0;
    } else if (last && threadIdx.x == 0) {
        if (OptTraits<OPT>::kPowers) {
            float p1 = h->b1p, p2 = h->b2p;
            for (int k = 0; k < applies; ++k) {
                p1 = __fmul_rn(p1, b1);
                p2 = __fmul_rn(p2, b2);
            }
            h->b1p = p1;
            h->b2p = p2;
        }
        h->step += applies;
        h->ticket = 0;
        const unsigned int seq = h->apply_seq + 1;
        __threadfence_system();
        publish_store(&h->apply_seq, seq);
        for (int c = 0; c < peers.n_mirror; ++c) publish_store(peers.mirror[c], seq);
        for (int c = 0; c < peers.n_mailbox; ++c) publish_add(peers.mailbox[c], 1u);
    }
}

// ---------------------------------------------------- request-free serving ----
// The reference's default discipline: every worker's push is applied when it
// ARRIVES and nobody waits for anybody (examples/mnist/mnist_replica.py:198-205,
// mnist.py:63-72) -- with no request from the worker.  Per batch of arrivals the PS runs
//     k_pick ; k_apply<.., PickSrc>
// issued by a host thread that polls the counter (psx_serve_start; psx.cu explains
// why the waits are not pre-enqueued on the stream).  A push bumps
// `arrivals`; the poll sees it; k_pick (one warp) looks at every slot flag,
// lists the slots holding an unconsumed push in the header and takes them off the
// counter; the apply kernel consumes exactly that list in ONE pass (in list order,
// each with its own beta powers: the serialisable async schedule) and its last CTA
// tells each consumed worker "your push k is in" (+ the global_step it produced)
// in that worker's own HBM.  The worker side is push ; stream-wait ; pull.
//
// SYNC (SyncReplicasOptimizer, mnist_replica.py:109-113,148-162): a gradient whose
// stamp (the global_step its parameters had) is older than the shard's global_step
// is dropped as stale; fresh ones wait as `pending` until R = replicas_to_aggregate
// of them are there; the first R in ARRIVAL order are averaged and applied once;
// every worker then receives a token (the chief's token queue), fast or slow.
template <int MODE>
__global__ void k_pick(ShardHeader *h, int n_slots, int aggregate)
{
    __shared__ unsigned int s_new[PSX_MAX_SLOTS];
    const int s = threadIdx.x;
    unsigned int seq = 0;
    bool fresh = false;
    if (s < n_slots) {
        seq = ld_sys(&h->slot_seq[s]);
        fresh = seq != h->slot_seen[s];
    }
    if (s < PSX_MAX_SLOTS) s_new[s] = fresh ? seq : 0u;
    __syncthreads();
    if (threadIdx.x != 0) return;
    unsigned int n_new = 0, n_pick = 0;
    if (MODE == PSX_MODE_ASYNC_ORDERED) {
        for (int k = 0; k < n_slots; ++k) {
            if (s_new[k] == 0u) continue;
            h->slot_seen[k] = s_new[k];
            h->pick[n_pick] = (unsigned int)k;
            h->pick_seq[n_pick] = s_new[k];
            ++n_pick;
            ++n_new;
        }
    } else {
        const unsigned int step = (unsigned int)h->step;
        for (int k = 0; k < n_slots; ++k) {
            if (s_new[k] != 0u) {               // a new push replaces whatever the slot held
                h->slot_seen[k] = s_new[k];
                h->pending[k] = 1u;
                h->arrival_rank[k] = ++h->arrival_ctr;
                ++n_new;
            }
            // stale: computed from parameters older than the current global_step
            if (h->pending[k] && (int)(ld_sys(&h->slot_stamp[k]) - step) < 0) {
                h->pending[k] = 0u;
                ++h->dropped;
            }
        }
        unsigned int n_pending = 0;
        for (int k = 0; k < n_slots; ++k) n_pending += h->pending[k];
        if (n_pending >= (unsigned int)aggregate) {
            for (int r = 0; r < aggregate; ++r) {          // the first R by arrival
                int best = -1;
                for (int k = 0; k < n_slots; ++k)
                    if (h->pending[k] && (best < 0 || (int)(h->arrival_rank[k] - h->arrival_rank[best]) < 0))
                        best = k;
                h->pending[best] = 0u;
                h->pick[n_pick] = (unsigned int)best;
                h->pick_seq[n_pick] = h->slot_seen[best];
                ++n_pick;
            }
        }
    }
    h->pick_n = n_pick;
    if (n_new) atomicSub(&h->arrivals, n_new);
}

// epilogue of a served apply: per-slot completion instead of the broadcast one
template <int OPT, int MODE>
__device__ __forceinline__ void finish_served(ShardHeader *h, int count, float b1, float b2)
{
    const bool last = last_cta<false>(&h->ticket);
    if (!last || threadIdx.x != 0) return;
    h->ticket = 0;
    if (count == 0) return;
    const int applies = (MODE == PSX_MODE_ASYNC_ORDERED) ? count : 1;
    if (OptTraits<OPT>::kPowers) {
        float p1 = h->b1p, p2 = h->b2p;
        for (int k = 0; k < applies; ++k) {
            p1 = __fmul_rn(p1, b1);
            p2 = __fmul_rn(p2, b2);
        }
        h->b1p = p1;
        h->b2p = p2;
    }
    const long long step0 = h->step;
    h->step = step0 + applies;
    h->served += (unsigned int)count;
    const unsigned int seq = h->apply_seq + 1;
    // the step values first, ONE system fence, then the words the workers wait on
    if (MODE == PSX_MODE_ASYNC_ORDERED) {
        for (int k = 0; k < count; ++k) {
            ClientBlock *cb = (ClientBlock *)h->client_block[h->pick[k]];
            if (cb) cb->step = step0 + k + 1;
        }
    } else {
        for (int c = 0; c < PSX_MAX_SLOTS; ++c) {
            ClientBlock *cb = (ClientBlock *)h->client_block[c];
            if (cb) cb->step = step0 + 1;
        }
    }
    __threadfence_system();
    publish_store(&h->apply_seq, seq);
    if (MODE == PSX_MODE_ASYNC_ORDERED) {
        for (int k = 0; k < count; ++k) {
            ClientBlock *cb = (ClientBlock *)h->client_block[h->pick[k]];
            if (cb) publish_store(&cb->applied, h->pick_seq[k]);
        }
    } else {
        for (int c = 0; c < PSX_MAX_SLOTS; ++c) {       // a token for EVERY worker
            ClientBlock *cb = (ClientBlock *)h->client_block[c];
            if (cb) publish_add(&cb->tokens, 1u);
        }
    }
}

constexpr int kApplyThreads = 256;
constexpr int kSlotChunk = 4;  // gradient vectors in flight per thread
#ifndef PSX_APPLY_MIN_CTAS
#define PSX_APPLY_MIN_CTAS 3   // resident CTAs per SM the register budget is cut for
#endif
#ifndef PSX_PREFETCH_STATE
#define PSX_PREFETCH_STATE 0   // 1: also request var/m/v of the next iteration early
#endif

// Where slot s's gradient vector i comes from.
template <typename WIRE> struct SlotSrc {            // landing slots in the shard
    static constexpr bool kPrefetch = false;         // local HBM: occupancy hides the latency
    const WIRE *base;
    size_t stride;                                   // elements between slots
    int first;
    __device__ __forceinline__ float4 load(int s, size_t i) const
    {
        return Vec4<WIRE>::load(base + (size_t)(first + s) * stride + 4 * i);
    }
};
template <typename WIRE> struct PeerSrc {            // bound worker buffers (peer HBM)
    static constexpr bool kPrefetch = true;          // NVLink round trip: prefetch one iteration
    using wire_t = WIRE;
    PeerSet peers;
    int first;
    __device__ __forceinline__ float4 load(int s, size_t i) const
    {
        return Vec4<WIRE>::load((const WIRE *)peers.grad[first + s] + 4 * i);
    }
};
// NVLS: ONE multicast address stands for the same range of EVERY worker's gradient
// buffer; multimem.ld_reduce makes the switch fetch all copies and return their
// f32 sum, so the kernel sees a single "slot" (count == 1) that already holds the
// W-way reduction.  The switch's summation order is its own: bit-exact against
// the oracle's slot order only for W <= 2 (a single commutative add), tolerance-
// checked beyond.
__device__ __forceinline__ float4 mc_ld_reduce(const float *mc)
{
    float4 v;
    asm volatile("multimem.ld_reduce.relaxed.sys.global.add.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
                 : "l"(mc)
                 : "memory");
    return v;
}
__device__ __forceinline__ void mc_st(float *mc, const float4 &v)
{
    asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(mc), "f"(v.x),
                 "f"(v.y), "f"(v.z), "f"(v.w)
                 : "memory");
}
// Served mode: which landing slots this apply consumes was decided by k_pick right
// before (same stream) and sits in the shard header.
template <typename WIRE> struct PickSrc {
    static constexpr bool kPrefetch = false;
    static constexpr bool kDynamic = true;
    const WIRE *base;
    size_t stride;
    const unsigned int *pick;        // set inside the kernel: the list, staged in shared memory
    __device__ __forceinline__ float4 load(int s, size_t i) const
    {
        return Vec4<WIRE>::load(base + (size_t)pick[s] * stride + 4 * i);
    }
};
template <typename SRC> struct IsDynamic { static constexpr bool value = false; };
template <typename W> struct IsDynamic<PickSrc<W>> { static constexpr bool value = true; };
template <typename SRC> struct WireOf { using type = float; };
template <typename W> struct WireOf<PeerSrc<W>> { using type = W; };
template <typename SRC> struct IsMulticast { static constexpr bool value = false; };

// Fused reduce + apply over a whole shard (n4 vectors).  SCATTER: also write
// the new parameters into every bound worker parameter buffer (psx_round).
template <int OPT, int MODE, bool SCATTER, typename SRC>
__global__ void __launch_bounds__(kApplyThreads, PSX_APPLY_MIN_CTAS)
k_apply(ShardHeader *__restrict__ h, float4 *__restrict__ var, float4 *__restrict__ mom,
        float4 *__restrict__ vel, SRC src, int count, size_t n4, PeerSet peers, int finish,
        unsigned int consume, int divisor)
{
    // count   = gradient sources read per element; served mode (PickSrc): whatever
    //           k_pick selected, read from the header (0 = nothing to do this time)
    // divisor = SYNC_MEAN's denominator (the number of workers aggregated)
    __shared__ unsigned int s_pick[PSX_MAX_SLOTS];
    if constexpr (IsDynamic<SRC>::value) {
        count = (int)h->pick_n;
        divisor = count;
        if (count == 0) n4 = 0;                 // nothing arrived that can be applied yet
        if (threadIdx.x < PSX_MAX_SLOTS) s_pick[threadIdx.x] = h->pick[threadIdx.x];
        src.pick = s_pick;
        __syncthreads();
    }
    // counted rendez-vous: the stream waited for arrivals >= consume right before
    // this launch; take them off the counter so the next round waits for the same
    // constant again (that is what makes a round replayable from a CUDA graph).
    // Next-round arrivals cannot come before this kernel's END (workers start their
    // next round only after it has bumped their mailbox), so this cannot race them.
    if (consume != 0 && blockIdx.x == 0 && threadIdx.x == 0) atomicSub(&h->arrivals, consume);
    __shared__ float s_alpha[PSX_MAX_SLOTS];
    const float lr = h->lr, b1 = h->b1, b2 = h->b2, eps = h->eps;
    const float omb1 = __fsub_rn(1.0f, b1);
    const float omb2 = __fsub_rn(1.0f, b2);
    if (OptTraits<OPT>::kPowers) {
        if (threadIdx.x == 0) {
            float p1 = h->b1p, p2 = h->b2p;
            const int na = (MODE == PSX_MODE_ASYNC_ORDERED) ? count : 1;
            for (int k = 0; k < na; ++k) {
                s_alpha[k] = adam_alpha(lr, p1, p2);
                p1 = __fmul_rn(p1, b1);
                p2 = __fmul_rn(p2, b2);
            }
        }
        __syncthreads();
    }
    const float fcount = (float)divisor;

    // Software pipeline: the first kSlotChunk gradient vectors of the NEXT
    // iteration are requested before this iteration's arithmetic.  With peer
    // sources (psx_round over NVLink, ~2-3.7 us per load) this doubles the bytes
    // each SM keeps in flight -- measured at N=2: 12 KB/SM in flight capped the
    // gather at ~615 GB/s (profiles/r02).
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    constexpr bool PF = SRC::kPrefetch;
    float4 gn[kSlotChunk];
    if (PF && i < n4) {
#pragma unroll
        for (int k = 0; k < kSlotChunk; ++k)
            if (k < count) gn[k] = src.load(k, i);
    }
#if PSX_PREFETCH_STATE
    float4 xn = make_float4(0.f, 0.f, 0.f, 0.f), mn = xn, vn = xn;
    if (i < n4) {
        xn = ld_stream(var + i);
        if (OptTraits<OPT>::kState >= 1) mn = ld_stream(mom + i);
        if (OptTraits<OPT>::kState >= 2) vn = ld_stream(vel + i);
    }
#endif
    for (; i < n4; i += stride) {
#if PSX_PREFETCH_STATE
        float4 x = xn, m = mn, v = vn;
        if (i + stride < n4) {
            xn = ld_stream(var + i + stride);
            if (OptTraits<OPT>::kState >= 1) mn = ld_stream(mom + i + stride);
            if (OptTraits<OPT>::kState >= 2) vn = ld_stream(vel + i + stride);
        }
#else
        float4 x = ld_stream(var + i);
        float4 m = make_float4(0.f, 0.f, 0.f, 0.f), v = m;
        if (OptTraits<OPT>::kState >= 1) m = ld_stream(mom + i);
        if (OptTraits<OPT>::kState >= 2) v = ld_stream(vel + i);
#endif
        float4 g[kSlotChunk];
        if (PF) {
#pragma unroll
            for (int k = 0; k < kSlotChunk; ++k) g[k] = gn[k];
            const size_t inext = i + stride;
            if (inext < n4) {
#pragma unroll
                for (int k = 0; k < kSlotChunk; ++k)
                    if (k < count) gn[k] = src.load(k, inext);
            }
        } else {
#pragma unroll
            for (int k = 0; k < kSlotChunk; ++k)
                if (k < count) g[k] = src.load(k, i);
        }
        float4 acc;
        for (int s0 = 0; s0 < count; s0 += kSlotChunk) {
            if (s0 > 0) {
#pragma unroll
                for (int k = 0; k < kSlotChunk; ++k)
                    if (s0 + k < count) g[k] = src.load(s0 + k, i);
            }
            if (MODE == PSX_MODE_ASYNC_ORDERED) {
#pragma unroll
                for (int k = 0; k < kSlotChunk; ++k)
                    if (s0 + k < count)
                        apply4<OPT>(x, m, v, g[k], lr, OptTraits<OPT>::kPowers ? s_alpha[s0 + k] : 0.f,
                                    b1, b2, omb1, omb2, eps);
            } else {
#pragma unroll
                for (int k = 0; k < kSlotChunk; ++k)
                    if (s0 + k < count) acc = (s0 + k == 0) ? g[k] : add4(acc, g[k]);
            }
        }
        if (MODE != PSX_MODE_ASYNC_ORDERED) {
            if (MODE == PSX_MODE_SYNC_MEAN) acc = div4(acc, fcount);
            apply4<OPT>(x, m, v, acc, lr, OptTraits<OPT>::kPowers ? s_alpha[0] : 0.f, b1, b2, omb1,
                        omb2, eps);
        }
        st_stream(var + i, x);
        if (OptTraits<OPT>::kState >= 1) st_stream(mom + i, m);
        if (OptTraits<OPT>::kState >= 2) st_stream(vel + i, v);
        if (SCATTER) {   // new parameters to every bound worker, cast to the wire dtype (RNE)
            using W = typename WireOf<SRC>::type;
            for (int s = 0; s < peers.n_param; ++s)
                Vec4<W>::store((W *)peers.param[s] + 4 * i, x);
        }
    }

    if (IsDynamic<SRC>::value)
        finish_served<OPT, MODE>(h, count, b1, b2);
    else
        finish_apply<OPT, IsMulticast<SRC>::value>(h, peers, (MODE == PSX_MODE_ASYNC_ORDERED) ? count : 1,
                                                    finish, b1, b2);
}

// ------------------------------------------------------------- NVLS round ----
// The one-kernel PS round with the NVSwitch doing both collective legs
// (psx_round on a shard bound with psx_round_bind_mc).  Per 16-byte vector of the
// shard's stripe:
//     g  = multimem.ld_reduce.add.v4.f32 [grad_mc + i]   switch fetches the vector from
//                                                        EVERY worker's gradient buffer
//                                                        and returns the f32 sum
//     the optimizer on var (+ its state arrays) in local HBM
//     multimem.st.v4.f32 [param_mc + i], var'            switch replicates the store into
//                                                        EVERY worker's parameter buffer
// NVLink bytes per GPU and direction for a bucket of B bytes striped over N GPUs:
// B (gradient copies leaving for the switch) + B/N (parameter stripe leaving) out,
// B/N (reduced stripe) + B (all stripes' parameters) in -- B(1 + 1/N) against the
// unicast kernel's 2(N-1)/N B.  The gather saturates the port's egress and the
// scatter its ingress, so they must overlap: each thread keeps the ld_reduce of
// its NEXT tile in flight while it applies and multicasts the current one.
constexpr int kMcThreads = 256;
#ifndef PSX_MC_UNROLL
#define PSX_MC_UNROLL 2            // vectors per thread and tile (ld_reduce in flight: 2x this)
#endif

template <int OPT, int MODE, int U>
__global__ void __launch_bounds__(kMcThreads, PSX_APPLY_MIN_CTAS)
k_round_mc(ShardHeader *__restrict__ h, float4 *__restrict__ var, float4 *__restrict__ mom,
           float4 *__restrict__ vel, const float *grad_mc, float *param_mc, size_t n4,
           PeerSet peers, unsigned int consume, int divisor)
{
    if (consume != 0 && blockIdx.x == 0 && threadIdx.x == 0) atomicSub(&h->arrivals, consume);
    const float lr = h->lr, b1 = h->b1, b2 = h->b2, eps = h->eps;
    const float omb1 = __fsub_rn(1.0f, b1);
    const float omb2 = __fsub_rn(1.0f, b2);
    const float alpha = OptTraits<OPT>::kPowers ? adam_alpha(lr, h->b1p, h->b2p) : 0.f;
    const float fdiv = (float)divisor;

    const size_t tile = (size_t)kMcThreads * U;
    const size_t tiles = (n4 + tile - 1) / tile;
    size_t t = blockIdx.x;
    float4 gn[U];
    if (t < tiles) {
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const size_t i = t * tile + (size_t)u * kMcThreads + threadIdx.x;
            if (i < n4) gn[u] = mc_ld_reduce(grad_mc + 4 * i);
        }
    }
    for (; t < tiles; t += gridDim.x) {
        float4 g[U], x[U], m[U], v[U];
        const size_t base = t * tile + threadIdx.x;
#pragma unroll
        for (int u = 0; u < U; ++u) {          // local state first: HBM latency overlaps the switch's
            const size_t i = base + (size_t)u * kMcThreads;
            if (i < n4) {
                x[u] = ld_stream(var + i);
                if (OptTraits<OPT>::kState >= 1) m[u] = ld_stream(mom + i);
                if (OptTraits<OPT>::kState >= 2) v[u] = ld_stream(vel + i);
            }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) g[u] = gn[u];
        const size_t tn = t + gridDim.x;
        if (tn < tiles) {
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const size_t i = tn * tile + (size_t)u * kMcThreads + threadIdx.x;
                if (i < n4) gn[u] = mc_ld_reduce(grad_mc + 4 * i);
            }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const size_t i = base + (size_t)u * kMcThreads;
            if (i < n4) {
                float4 acc = g[u];
                if (MODE == PSX_MODE_SYNC_MEAN) acc = div4(acc, fdiv);
                apply4<OPT>(x[u], m[u], v[u], acc, lr, alpha, b1, b2, omb1, omb2, eps);
                st_stream(var + i, x[u]);
                if (OptTraits<OPT>::kState >= 1) st_stream(mom + i, m[u]);
                if (OptTraits<OPT>::kState >= 2) st_stream(vel + i, v[u]);
                mc_st(param_mc + 4 * i, x[u]);
            }
        }
    }
    finish_apply<OPT, true>(h, peers, 1, 1, b1, b2);
}

// ---------------------------------------------- index-list (sparse) rows ----
// IndexedSlices push for embedding-like variables (SURVEY 8f-3): a worker ships
// K rows of length D plus their row indices instead of the dense gradient.  The
// rows land in the worker's OWN landing slot, which is laid out for this as
//     [ count u64 | pad | idx i64[K] | pad to 16 B | rows wire[K x D] ]
// Indices must be strictly ascending (unique): the worker de-duplicates its own
// slices (TF does the same before a sparse Adam apply); duplicates ACROSS workers
// are merged on the PS in worker order, found by binary search -- no sort, no
// atomics on floats, bit-reproducible.
struct RowsHeader {
    unsigned long long count;
    unsigned long long row_len;
};
__host__ __device__ inline size_t rows_idx_off() { return 16; }
__host__ __device__ inline size_t rows_data_off(size_t k) { return (16 + k * 8 + 15) / 16 * 16; }

template <typename SRC, typename DST>
__global__ void __launch_bounds__(kCopyThreads)
k_push_rows(char *slot, const long long *__restrict__ idx, const SRC *__restrict__ rows, size_t k,
            size_t d, unsigned int *ticket, unsigned int *flag, unsigned int *arrivals,
            unsigned int seq)
{
    long long *didx = (long long *)(slot + rows_idx_off());
    DST *drows = (DST *)(slot + rows_data_off(k));
    const size_t tid = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t nth = (size_t)gridDim.x * blockDim.x;
    for (size_t i = tid; i < k; i += nth) didx[i] = idx[i];
    for (size_t i = tid; i < k * d; i += nth) drows[i] = from_f32<DST>(to_f32<SRC>(rows[i]));
    if (tid == 0) {
        RowsHeader *rh = (RowsHeader *)slot;
        rh->count = k;
        rh->row_len = d;
    }
    if (last_cta(ticket) && threadIdx.x == 0) {
        *ticket = 0;
        __threadfence_system();
        publish_store(flag, seq);
        publish_add_release(arrivals, 1u);
    }
}

__device__ __forceinline__ long long rows_find(const long long *idx, long long n, long long key)
{
    long long lo = 0, hi = n;
    while (lo < hi) {
        long long mid = (lo + hi) >> 1;
        if (idx[mid] < key) lo = mid + 1;
        else hi = mid;
    }
    return (lo < n && idx[lo] == key) ? lo : -1;
}

// One warp per pushed entry (slot w, position k).  The entry whose worker is the
// LOWEST one holding that row index is the row's representative: it sums the
// row's contributions in worker order ((g_w + g_w') + ...), divides for MEAN, and
// applies the optimizer to that row of var (m, v) only -- untouched rows keep their
// value and their state ("lazy" sparse semantics, TF's SparseApply*).
template <int OPT, int MODE, typename WIRE>
__global__ void __launch_bounds__(256)
k_apply_rows(ShardHeader *__restrict__ h, float *__restrict__ var, float *__restrict__ mom,
             float *__restrict__ vel, const char *slots, size_t slot_stride, int first, int count,
             size_t d, size_t n_rows, PeerSet peers)
{
    const float lr = h->lr, b1 = h->b1, b2 = h->b2, eps = h->eps;
    const float omb1 = __fsub_rn(1.0f, b1), omb2 = __fsub_rn(1.0f, b2);
    const float alpha = OptTraits<OPT>::kPowers ? adam_alpha(lr, h->b1p, h->b2p) : 0.f;
    const float fcount = (float)count;
    const int lane = threadIdx.x & 31;
    const size_t warp = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const size_t n_warps = ((size_t)gridDim.x * blockDim.x) >> 5;
    // entries are numbered slot-major: prefix over the slots' counts
    size_t total = 0;
    for (int s = 0; s < count; ++s)
        total += ((const RowsHeader *)(slots + (size_t)(first + s) * slot_stride))->count;
    for (size_t e = warp; e < total; e += n_warps) {
        int w = 0;
        size_t k = e;
        for (;; ++w) {
            const size_t c = ((const RowsHeader *)(slots + (size_t)(first + w) * slot_stride))->count;
            if (k < c) break;
            k -= c;
        }
        const char *sw = slots + (size_t)(first + w) * slot_stride;
        const size_t kw = ((const RowsHeader *)sw)->count;
        const long long row = ((const long long *)(sw + rows_idx_off()))[k];
        if (row < 0 || (size_t)row >= n_rows) continue;          // out of range: ignored
        bool rep = true;                                          // lowest worker holding `row`?
        for (int w2 = 0; w2 < w && rep; ++w2) {
            const char *s2 = slots + (size_t)(first + w2) * slot_stride;
            if (rows_find((const long long *)(s2 + rows_idx_off()),
                          (long long)((const RowsHeader *)s2)->count, row) >= 0)
                rep = false;
        }
        if (!rep) continue;
        long long pos[PSX_MAX_SLOTS];
        for (int w2 = w + 1; w2 < count; ++w2) {
            const char *s2 = slots + (size_t)(first + w2) * slot_stride;
            pos[w2] = rows_find((const long long *)(s2 + rows_idx_off()),
                                (long long)((const RowsHeader *)s2)->count, row);
        }
        const WIRE *g0 = (const WIRE *)(sw + rows_data_off(kw)) + k * d;
        for (size_t j = lane; j < d; j += 32) {
            float g = to_f32<WIRE>(g0[j]);
            for (int w2 = w + 1; w2 < count; ++w2) {
                if (pos[w2] < 0) continue;
                const char *s2 = slots + (size_t)(first + w2) * slot_stride;
                const size_t k2 = ((const RowsHeader *)s2)->count;
                g = __fadd_rn(g, to_f32<WIRE>(((const WIRE *)(s2 + rows_data_off(k2)))[(size_t)pos[w2] * d + j]));
            }
            if (MODE == PSX_MODE_SYNC_MEAN) g = __fdiv_rn(g, fcount);
            const size_t at = (size_t)row * d + j;
            float x = var[at], m = 0.f, v = 0.f;
            if (OptTraits<OPT>::kState >= 1) m = mom[at];
            if (OptTraits<OPT>::kState >= 2) v = vel[at];
            apply1<OPT>(x, m, v, g, lr, alpha, b1, b2, omb1, omb2, eps);
            if (OptTraits<OPT>::kState >= 1) mom[at] = m;
            if (OptTraits<OPT>::kState >= 2) vel[at] = v;
            var[at] = x;
        }
    }
    finish_apply<OPT, false>(h, peers, 1, 1, b1, b2);
}

}  // namespace psx
