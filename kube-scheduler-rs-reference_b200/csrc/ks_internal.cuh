// ks_internal.cuh — shared device-side views, PTX helpers and launch plumbing (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>

#include "../../include/ksched.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "libksched is written for sm_100a (B200) only"
#endif

namespace ks {

constexpr int TILE_N = 1024;        // nodes per shared-memory tile of the direct kernel
constexpr int DIRECT_THREADS = 256; // 8 warps

// Device-resident node table (SoA, padded to a multiple of TILE_N with never-feasible sentinels:
// free = INT64_MIN, labels = 0).  labels are word-major: labels[w*Npad + n].
struct NodeTable {
    const int64_t* free_cpu;
    const int64_t* free_mem;
    const int64_t* alloc_cpu;
    const int64_t* alloc_mem;
    const uint64_t* labels;
    uint32_t N, Npad, W;
};

struct PodView {
    const int64_t* req_cpu;
    const int64_t* req_mem;
    const uint64_t* sel; // row-major [P*W]
    uint32_t P;
};

struct OutView {
    int32_t* node_idx;
    int64_t* score;
    uint32_t* cnt;
    uint32_t* mask;          // may be nullptr
    uint64_t mask_row_words; // row pitch in 32-bit words
    uint32_t mask_valid_words; // words per row that may be written: 8*ceil(N/256)
};

// Fused all-gather of the bindings (ks_exchange, include/ksched.h): peer-mapped destinations of this rank's shard
struct PeerOut {
    uint32_t n = 0; // peers; 0 = no exchange
    uint32_t world = 1, rank = 0;
    int32_t* idx[KS_MAX_PEERS];
    int64_t* score[KS_MAX_PEERS];
    uint32_t* flag[KS_MAX_PEERS];
    uint32_t* local_flags = nullptr;
    uint32_t* state = nullptr; // [0] = step sequence number, [1] = CTA completion counter, [2..11] = stamps (below)
};

// Diagnostic trace of the last exchange step: %globaltimer (ns) of 0 = first argmax CTA started, 1 = flags published,
// 2 = wait kernel started, 3 = wait kernel saw every peer, 4 = first CTA of the tail kernel started.  Five 64-bit words
// after the two state words.
__device__ __forceinline__ void exchange_stamp(const PeerOut& po, int which) {
    if (po.n == 0) return;
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    reinterpret_cast<volatile unsigned long long*>(po.state + 2)[which] = t;
}

// Last CTA of the kernel that completes this rank's bindings: publish a new sequence number to every peer.
// Call at the very end of the kernel, by all threads of the CTA.
__device__ __forceinline__ void exchange_signal(const PeerOut& po) {
    if (po.n == 0) return;
    __syncthreads(); // every store of this CTA has been issued
    if (threadIdx.x == 0) {
        __threadfence_system(); // ... and is visible system-wide before the counter moves
        const uint32_t ctas = gridDim.x * gridDim.y * gridDim.z;
        if (atomicAdd(po.state + 1, 1u) == ctas - 1) {
            po.state[1] = 0; // every CTA has arrived: ready for the next launch
            const uint32_t seq = po.state[0] + 1;
            po.state[0] = seq;
            exchange_stamp(po, 1);
            __threadfence_system();
            for (uint32_t k = 0; k < po.n; k++)
                asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(po.flag[k]), "r"(seq) : "memory");
            asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(po.local_flags + po.rank), "r"(seq) : "memory");
        }
    }
}

// Per-(chunk,pod) partial results when the node dimension is split across CTAs (small P).
struct PartialView {
    int64_t* key;  // best policy key (LEFTOVER: node priority; LEAST_ALLOCATED: score)
    int32_t* idx;
    uint32_t* cnt;
};

// ---- what a cell's result means ------------------------------------------------------------------------------------
// The one device-side definition of the score policies (KS_SCORE_* in include/ksched.h), the argmax rule, claim
// resolution and the binding store; oracle/oracle.c is the same definition on the CPU and the tests compare the two bit
// for bit.  Feasibility is predicates.rs:42 (fit, non-strict) and :45-61 (selector); the reference itself has no score.
// Free, allocatable and requested values are range-checked at snapshot time (KS_MAX_CPU_MILLI, KS_MAX_MEM_BYTES), so
// no term below leaves int64.

// KS_SCORE_LEFTOVER = leftover_prio(free) - leftover_cost(request): separable, so a node's rank does not depend on the
// pod and the argmax keys are node priorities.  The unsigned shift is free_cpu * 2^22 without signed-overflow UB.
__device__ __forceinline__ int64_t leftover_prio(int64_t fc, int64_t fm) {
    return (int64_t)(((uint64_t)fc << 22) + (uint64_t)fm);
}
__device__ __forceinline__ int64_t leftover_cost(int64_t rc, int64_t rm) { return leftover_prio(rc, rm); }

// KS_SCORE_LEAST_ALLOCATED: mean of the cpu and memory percentages left after the request, truncating divisions as in
// C and Rust; a resource with allocatable <= 0 contributes 0.  Not separable: the argmax keys are the scores themselves.
__device__ __forceinline__ int64_t least_alloc_score(int64_t fc, int64_t fm, int64_t ac, int64_t am, int64_t rc, int64_t rm) {
    const int64_t pc = ac > 0 ? ((fc - rc) * 100) / ac : 0;
    const int64_t pm = am > 0 ? ((fm - rm) * 100) / am : 0;
    return (pc + pm) / 2;
}

// The score a binding reports for the winning argmax key of a pod with request (rc, rm).
__device__ __forceinline__ int64_t key_to_score(int policy, int64_t key, int64_t rc, int64_t rm) {
    return policy == KS_SCORE_LEFTOVER ? key - leftover_cost(rc, rm) : key;
}

// The argmax rule: the larger key wins, equal keys go to the lower node index; idx < 0 means "no feasible node" and
// never wins.
__device__ __forceinline__ bool argmax_better(int64_t key, int32_t idx, int64_t best_key, int32_t best_idx) {
    return idx >= 0 && (best_idx < 0 || key > best_key || (key == best_key && idx < best_idx));
}

struct Candidate {
    int64_t key;
    int32_t idx;
};

// Merges the (key, idx) candidates of the 32 lanes by argmax_better; every lane gets the warp's winner.  Taken and
// returned by value: reference parameters would make the caller's running best address-taken, and the compiler then
// stops turning the caller's own compare-and-update into selects.
__device__ __forceinline__ Candidate warp_argmax(int64_t key, int32_t idx) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        const int64_t ok = __shfl_xor_sync(0xffffffffu, key, off);
        const int32_t oi = __shfl_xor_sync(0xffffffffu, idx, off);
        if (argmax_better(ok, oi, key, idx)) {
            key = ok;
            idx = oi;
        }
    }
    return {key, idx};
}

// Claims against node capacity (streaming reconcile, include/ksched.h): the claims on one node are taken in arrival
// order, each accepted iff its request still fits what the accepted claims before it left (predicates.rs:42), and the
// accepted requests are committed to free[] (util.rs:31-36).  The caller has set keys[k] = node << 32 | k for every
// claim k < n that names a node and keys[k] = ~0 for the others; keys must have room for n rounded up to a power of
// two.  One CTA of THREADS threads (every thread calls this) sorts the keys (bitonic, shared memory), then one thread
// per node segment walks it: a single writer per node, no atomics, deterministic.  request(k) returns claim k's (cpu,
// memory); record(k, ok) is called once for every claim that names a node.  free[] is read through L2 because
// k_stream_batch calls this after other CTAs of the same launch have written it.
template <uint32_t THREADS, class Request, class Record>
__device__ __forceinline__ void resolve_claims(unsigned long long* keys, uint32_t n, int64_t* free_cpu, int64_t* free_mem,
                                               Request request, Record record) {
    uint32_t m = 1;
    while (m < n) m <<= 1;
    for (uint32_t i = n + threadIdx.x; i < m; i += THREADS) keys[i] = ~0ull; // padding sorts last
    __syncthreads();
    for (uint32_t size = 2; size <= m; size <<= 1)
        for (uint32_t stride = size >> 1; stride > 0; stride >>= 1) {
            for (uint32_t i = threadIdx.x; i < m / 2; i += THREADS) {
                const uint32_t lo = 2 * i - (i & (stride - 1)), hi = lo + stride;
                const bool up = (lo & size) == 0;
                const unsigned long long a = keys[lo], b = keys[hi];
                if ((a > b) == up) {
                    keys[lo] = b;
                    keys[hi] = a;
                }
            }
            __syncthreads();
        }
    for (uint32_t i = threadIdx.x; i < m; i += THREADS) {
        const unsigned long long key = keys[i];
        if (key == ~0ull) continue;
        const uint32_t node = (uint32_t)(key >> 32);
        if (i > 0 && (uint32_t)(keys[i - 1] >> 32) == node) continue; // not a segment head
        int64_t fc = __ldcg(free_cpu + node), fm = __ldcg(free_mem + node);
        for (uint32_t j = i; j < m && keys[j] != ~0ull && (uint32_t)(keys[j] >> 32) == node; j++) {
            const uint32_t k = (uint32_t)keys[j];
            const longlong2 r = request(k);
            const bool ok = r.x <= fc && r.y <= fm;
            record(k, ok);
            if (ok) {
                fc -= r.x;
                fm -= r.y;
            }
        }
        free_cpu[node] = fc;
        free_mem[node] = fm;
    }
}

// Stores pod p's binding into the local outputs the caller asked for and, with a fused exchange, into every peer's
// gather buffer.
__device__ __forceinline__ void store_binding(const OutView& ov, const PeerOut& po, uint32_t p, int32_t idx, int64_t score) {
    if (ov.node_idx) ov.node_idx[p] = idx;
    if (ov.score) ov.score[p] = score;
    for (uint32_t k = 0; k < po.n; k++) {
        po.idx[k][p] = idx;
        po.score[k][p] = score;
    }
}

extern std::atomic<uint64_t> g_launches;

// ---- PTX helpers: mbarrier + 1-D TMA bulk copy (cp.async.bulk -> SASS UBLKCP) ----
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_mbar_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra WAIT_DONE;\n\t"
        "bra WAIT_LOOP;\n\t"
        "WAIT_DONE:\n\t"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
// global -> shared bulk copy, completion signalled on an mbarrier (bytes multiple of 16, 16B-aligned)
__device__ __forceinline__ void tma_bulk_g2s(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(smem_dst)),
                 "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

// ---- launch-side plumbing shared by the API and the kernel files ----
struct SelectLaunch {
    NodeTable nt;
    PodView pv;
    OutView ov;
    int policy;
    cudaStream_t stream;
    // host-space outputs: when set, the launcher may copy these results back as soon as they exist (the bindings
    // are ready long before the mask kernel ends) and clears the pointer it has served
    int32_t* host_node_idx = nullptr;
    int64_t* host_score = nullptr;
    cudaEvent_t ready_event = nullptr; // caller's "bindings are final" event (ks_bindings.bindings_ready_event)
    PeerOut po;                        // fused all-gather of the bindings (po.n == 0: none)
};

// Records the caller's ready event on st.  Inside a stream capture it must become an external event node: a plain record
// would only order nodes inside the graph and never signal the caller's event on replay.
inline cudaError_t record_ready_event(cudaEvent_t ev, cudaStream_t st) {
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    const cudaError_t e = cudaStreamIsCapturing(st, &cs);
    if (e != cudaSuccess) return e;
    return cudaEventRecordWithFlags(ev, st, cs == cudaStreamCaptureStatusActive ? cudaEventRecordExternal : cudaEventRecordDefault);
}

} // namespace ks
