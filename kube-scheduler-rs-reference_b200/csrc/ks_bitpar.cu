// ks_bitpar.cu — bit-parallel fused feasibility pass for sm_100a (design notes in ks_bitpar.h, DESIGN.md).
//
//   per snapshot   k_node_bound, k_node_splitters/_bucket/_scatter/_rank  sample sort: global position of every node in
//                                   free_cpu / free_mem / leftover-priority / least-allocated-bound order
//                  k_build_cbtile   per column block (8 tiles of 256 nodes, node-index order): octet-interleaved prefix
//                                   tables + label-pair columns, staged in shared memory by the mask kernel
//                  k_build_ranks    rank tables: tile-local rank of every possible threshold (read through L1/L2)
//                  k_build_tile     flat indexes in priority order / bound order for the argmax kernels
//   per call       k_pod_ranks      request -> global rank threshold (splitters in smem + short global search) and the mask
//                                   kernel's 16-byte pod record, in pod order
//                  k_mask_rows      persistent, 1 CTA per SM; table blob staged by TMA bulk copies (cp.async.bulk + mbarrier);
//                                   8 lanes = the 8 tiles of one pod: rank load -> 2 table rows (+ label columns) -> AND ->
//                                   one 256-bit store per lane; counts by shuffle + one RED per pod and column block
//                  k_first_fit_head/_tail  argmax KS_SCORE_LEFTOVER = first feasible node in priority order (early exit)
//                  k_least_alloc    argmax KS_SCORE_LEAST_ALLOCATED: bound-ordered scan, exact scores, early exit
// Semantics per cell are exactly predicates.rs:42 / :45-61 (see include/ksched.h); only the evaluation
// order differs, and every output is compared bit-for-bit with the oracle in tests/.
#include "ks_bitpar.h"

#include <algorithm>
#include <cstdlib>
#include <cstring>

namespace ks {

// ------------------------------------------------------------------------------------------------ step trace
// KS_TRACE=1 (environment, read when the index is created): every kernel of a select stamps %globaltimer into a small
// device buffer - first CTA at its start, every CTA at its end (atomic max) - so that the timeline of one step can be read
// back with ks_last_trace (nsys is not available on the target boxes and ncu serialises the streams).  Off: one
// constant-bank load per CTA.
__constant__ unsigned long long* c_trace = nullptr;
enum TraceSlot : int {
    TR_RANKS_START = 0, TR_RANKS_END, TR_ARGMAX1_START, TR_ARGMAX1_END, TR_ARGMAX2_START, TR_ARGMAX2_END,
    TR_MASK_START, TR_MASK_END, TR_MASK_FIRST_CTA_END_INV, TR_SLOTS
};
__device__ __forceinline__ unsigned long long global_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
// call with one thread per CTA
__device__ __forceinline__ void trace_start(int slot) {
    unsigned long long* tr = c_trace;
    if (tr && blockIdx.x == 0) tr[slot] = global_ns();
}
__device__ __forceinline__ void trace_end(int slot) {
    unsigned long long* tr = c_trace;
    if (tr) atomicMax(tr + slot, global_ns());
}

// ------------------------------------------------------------------------------------------------ build
// ---- node ranking: sample sort ------------------------------------------------------------------------------
// Three total orders over the N nodes are needed: ascending free_cpu, ascending free_mem, descending priority,
// ties always by node index.  All three are "ascending (v', index)" with v' = free_cpu, free_mem, -priority.
// k_node_splitters sorts 1024 sampled keys per order in shared memory and keeps 255 splitters; k_node_bucket drops
// every node into one of 256 buckets per order; k_node_rank counts, inside the bucket only, the keys below the
// node's own: position = bucket start + that count.  O(N * (log 256 + N/256)) instead of O(N^2).
struct NodeKey {
    int64_t v;
    uint32_t idx;
};
__device__ __forceinline__ bool key_less(int64_t av, uint32_t ai, int64_t bv, uint32_t bi) {
    return av < bv || (av == bv && ai < bi);
}
// KS_SCORE_LEAST_ALLOCATED bound: the score of node n for a pod that requests nothing.  For requests >= 0 the score of
// every feasible (pod, n) cell is <= least_alloc_bound(n) (same truncating divisions, monotone in the numerators).
__device__ __forceinline__ int64_t least_alloc_bound(const NodeTable& nt, uint32_t n) {
    return least_alloc_score(nt.free_cpu[n], nt.free_mem[n], nt.alloc_cpu[n], nt.alloc_mem[n], 0, 0);
}
// prio[0..Npad) = leftover priority, prio[Npad..Npad+N) = least-allocated bound (k_node_bound, once per build)
__device__ __forceinline__ int64_t order_value(const NodeTable& nt, const int64_t* __restrict__ prio, int k, uint32_t n) {
    return k == 0 ? nt.free_cpu[n] : (k == 1 ? nt.free_mem[n] : (k == 2 ? -prio[n] : -prio[(size_t)nt.Npad + n]));
}

// least-allocated bound of every node + which label bits some node carries (a selector naming a dead bit is
// infeasible everywhere: the argmax kernels answer it without scanning)
__global__ void __launch_bounds__(256) k_node_bound(NodeTable nt, int64_t* __restrict__ bound, unsigned long long* __restrict__ live) {
    const uint32_t n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= nt.N) return;
    bound[n] = least_alloc_bound(nt, n);
    long long* amax = reinterpret_cast<long long*>(live + KS_MAX_LABEL_WORDS); // [2]: max allocatable cpu, memory
    if (nt.alloc_cpu[n] > __ldcg(amax)) atomicMax(amax, (long long)nt.alloc_cpu[n]);
    if (nt.alloc_mem[n] > __ldcg(amax + 1)) atomicMax(amax + 1, (long long)nt.alloc_mem[n]);
    for (uint32_t w = 0; w < nt.W; w++) {
        const unsigned long long v = nt.labels[(size_t)w * nt.Npad + n];
        if (v & ~__ldcg(live + w)) atomicOr(live + w, v);
    }
}

constexpr int RANK_SAMPLES = 1024, RANK_BUCKETS = 256;
// Work cursors of k_mask_rows (one per column block), zeroed by k_pod_ranks.  One cursor per 128-byte line: with all cursors in one line the L2 serialised every claim of the whole chip on it
// (~3 ns each: 781k claims = the whole 2.4 ms the kernel then took at C3, whatever the block size).
constexpr uint32_t RW_CURSOR_STRIDE = 32;
// Splitters per resource in k_pod_ranks' shared memory (dynamic, 16 bytes per splitter pair: <= 128 KB).  With 8192 the part
// of a search that is left for the sorted array in L2 covers <= 7 elements of one 64-byte block (C3: stride 8): ~1.6 random
// 32-byte sector requests per search instead of ~4 with 2048 splitters - and that request rate is what bounds the kernel.
constexpr int RANK_SPLITTERS = 8192;
constexpr int RANK_THREADS = 1024; // one CTA per SM
constexpr int N_ORDERS = 4; // free_cpu, free_mem, leftover priority, least-allocated bound

__global__ void __launch_bounds__(RANK_SAMPLES)
    k_node_splitters(NodeTable nt, const int64_t* __restrict__ prio, int64_t* __restrict__ spl_v,
                     uint32_t* __restrict__ spl_i, uint32_t* __restrict__ hist) {
    __shared__ int64_t s_v[RANK_SAMPLES];
    __shared__ uint32_t s_i[RANK_SAMPLES];
    const uint32_t t = threadIdx.x, k = blockIdx.x; // one CTA per order
    const uint32_t n = (uint32_t)(((uint64_t)t * nt.N) / RANK_SAMPLES);
    s_v[t] = order_value(nt, prio, k, n);
    s_i[t] = n;
    if (t < RANK_BUCKETS) hist[k * RANK_BUCKETS + t] = 0;
    __syncthreads();
    for (uint32_t size = 2; size <= RANK_SAMPLES; size <<= 1)
        for (uint32_t stride = size >> 1; stride > 0; stride >>= 1) {
            if (t < RANK_SAMPLES / 2) {
                const uint32_t lo = 2 * t - (t & (stride - 1)), hi = lo + stride;
                const bool up = (lo & size) == 0;
                const int64_t av = s_v[lo], bv = s_v[hi];
                const uint32_t ai = s_i[lo], bi = s_i[hi];
                if (key_less(bv, bi, av, ai) == up) {
                    s_v[lo] = bv; s_i[lo] = bi;
                    s_v[hi] = av; s_i[hi] = ai;
                }
            }
            __syncthreads();
        }
    if (t < RANK_BUCKETS - 1) { // splitter j = sample 4(j+1)-1
        spl_v[k * RANK_BUCKETS + t] = s_v[4 * (t + 1) - 1];
        spl_i[k * RANK_BUCKETS + t] = s_i[4 * (t + 1) - 1];
    }
}

__global__ void __launch_bounds__(256)
    k_node_bucket(NodeTable nt, const int64_t* __restrict__ prio, const int64_t* __restrict__ spl_v,
                  const uint32_t* __restrict__ spl_i, uint32_t* __restrict__ hist, uint8_t* __restrict__ bkt,
                  uint32_t* __restrict__ loc) {
    __shared__ int64_t s_v[N_ORDERS][RANK_BUCKETS];
    __shared__ uint32_t s_i[N_ORDERS][RANK_BUCKETS];
    for (uint32_t j = threadIdx.x; j < N_ORDERS * (RANK_BUCKETS - 1); j += blockDim.x) {
        const uint32_t k = j / (RANK_BUCKETS - 1), q = j % (RANK_BUCKETS - 1);
        s_v[k][q] = spl_v[k * RANK_BUCKETS + q];
        s_i[k][q] = spl_i[k * RANK_BUCKETS + q];
    }
    __syncthreads();
    const uint32_t n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= nt.N) return;
#pragma unroll
    for (int k = 0; k < N_ORDERS; k++) {
        const int64_t v = order_value(nt, prio, k, n);
        uint32_t lo = 0, len = RANK_BUCKETS - 1; // number of splitters < key
        while (len > 0) {
            const uint32_t half = len >> 1;
            if (key_less(s_v[k][lo + half], s_i[k][lo + half], v, n)) {
                lo += half + 1;
                len -= half + 1;
            } else {
                len = half;
            }
        }
        bkt[(size_t)k * nt.N + n] = (uint8_t)lo;
        loc[(size_t)k * nt.N + n] = atomicAdd(&hist[k * RANK_BUCKETS + lo], 1u);
    }
}

// bucket-ordered node lists (order inside a bucket is arbitrary; k_node_rank fixes the final positions)
__global__ void __launch_bounds__(256)
    k_node_scatter(uint32_t N, const uint32_t* __restrict__ hist, const uint8_t* __restrict__ bkt,
                   const uint32_t* __restrict__ loc, uint32_t* __restrict__ perm) {
    __shared__ uint32_t s_start[N_ORDERS][RANK_BUCKETS];
    if (threadIdx.x < N_ORDERS) {
        uint32_t acc = 0;
        for (int b = 0; b < RANK_BUCKETS; b++) {
            s_start[threadIdx.x][b] = acc;
            acc += hist[threadIdx.x * RANK_BUCKETS + b];
        }
    }
    __syncthreads();
    const uint32_t n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
#pragma unroll
    for (int k = 0; k < N_ORDERS; k++)
        perm[(size_t)k * N + s_start[k][bkt[(size_t)k * N + n]] + loc[(size_t)k * N + n]] = n;
}

__global__ void __launch_bounds__(256)
    k_node_rank(NodeTable nt, const int64_t* __restrict__ prio, const uint32_t* __restrict__ hist,
                const uint8_t* __restrict__ bkt, const uint32_t* __restrict__ perm, int64_t* __restrict__ sortedC,
                int64_t* __restrict__ sortedM, uint32_t* __restrict__ gposC, uint32_t* __restrict__ gposM,
                int64_t* __restrict__ ord_prio, int32_t* __restrict__ ord_idx, uint32_t Nord,
                int64_t* __restrict__ splC, int64_t* __restrict__ splM, uint32_t spl_stride,
                int64_t* __restrict__ ordL_s0, int32_t* __restrict__ ordL_idx) {
    __shared__ uint32_t s_start[N_ORDERS][RANK_BUCKETS + 1];
    if (threadIdx.x < N_ORDERS) {
        uint32_t acc = 0;
        for (int b = 0; b < RANK_BUCKETS; b++) {
            s_start[threadIdx.x][b] = acc;
            acc += hist[threadIdx.x * RANK_BUCKETS + b];
        }
        s_start[threadIdx.x][RANK_BUCKETS] = acc;
    }
    __syncthreads();
    const uint32_t n = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t N = nt.N;
    if (n < N) {
        uint32_t pos[N_ORDERS];
#pragma unroll
        for (int k = 0; k < N_ORDERS; k++) {
            const int64_t v = order_value(nt, prio, k, n);
            const uint32_t b = bkt[(size_t)k * N + n];
            uint32_t c = 0;
            for (uint32_t j = s_start[k][b]; j < s_start[k][b + 1]; j++) {
                const uint32_t m = perm[(size_t)k * N + j];
                c += key_less(order_value(nt, prio, k, m), m, v, n);
            }
            pos[k] = s_start[k][b] + c;
        }
        const int64_t fc = nt.free_cpu[n], fm = nt.free_mem[n];
        gposC[n] = pos[0];
        gposM[n] = pos[1];
        sortedC[pos[0]] = fc;
        sortedM[pos[1]] = fm;
        if (pos[0] % spl_stride == 0) splC[pos[0] / spl_stride] = fc;
        if (pos[1] % spl_stride == 0) splM[pos[1] / spl_stride] = fm;
        ord_prio[pos[2]] = prio[n];
        ord_idx[pos[2]] = (int32_t)n;
        ordL_s0[pos[3]] = prio[(size_t)nt.Npad + n];
        ordL_idx[pos[3]] = (int32_t)n;
    } else if (n < Nord) { // padding of the priority / bound orders
        ord_prio[n] = INT64_MIN;
        ord_idx[n] = -1;
        ordL_s0[n] = INT64_MIN;
        ordL_idx[n] = -1;
    }
}

static uint32_t pair_stride(uint32_t nt) { return nt * 32u; }

// Prefix tables are interleaved by QUADS of tiles: row r of tiles 4k..4k+3 forms one 128-byte line
//   [tile 4k row r | tile 4k+1 row r | tile 4k+2 row r | tile 4k+3 row r]
// so the four tiles that the 8 lanes of a shared-memory phase work on always sit in four different pairs of 16-byte
// bank groups, whatever their (unrelated) ranks are.  Byte offset of (tile, row) inside a table area:
__host__ __device__ __forceinline__ uint32_t table_row_offset(uint32_t tile, uint32_t row) {
    return (tile >> 2) * (uint32_t)(BP_ROWS * 128) + row * 128u + (tile & 3u) * 32u;
}
__host__ __device__ __forceinline__ uint32_t table_area_bytes(uint32_t nt) { return ((nt + 3u) / 4u) * (uint32_t)(BP_ROWS * 128); }

// One CTA builds the index of one 256-slot tile.  slot_node maps slot -> node (nullptr = identity, i.e. the
// node-index order used for the mask; ord_idx = priority order used for the argmax).
__global__ void __launch_bounds__(288)
    k_build_tile(NodeTable nt, const uint32_t* __restrict__ gposC, const uint32_t* __restrict__ gposM,
                 const int32_t* __restrict__ slot_node, uint8_t* __restrict__ blob, BitparLayout lay) {
    __shared__ uint32_t s_g[2][BP_TILE];
    __shared__ uint16_t s_lr[2][BP_TILE];
    __shared__ uint8_t s_valid[BP_TILE];
    __shared__ uint64_t s_lab[KS_MAX_LABEL_WORDS][BP_TILE];
    const uint32_t tile_g = blockIdx.x, cb = tile_g / lay.nt, t = tile_g % lay.nt, s = threadIdx.x;
    uint8_t* B = blob + (size_t)cb * lay.blob_bytes;
    if (s < BP_TILE) {
        const uint32_t slot = tile_g * BP_TILE + s;
        const bool v = slot < nt.N;
        const uint32_t n = v ? (slot_node ? (uint32_t)slot_node[slot] : slot) : 0;
        s_valid[s] = v;
        s_g[0][s] = v ? gposC[n] : 0xFFFFFFFFu;
        s_g[1][s] = v ? gposM[n] : 0xFFFFFFFFu;
        for (uint32_t w = 0; w < nt.W; w++) s_lab[w][s] = v ? nt.labels[(size_t)w * nt.Npad + n] : 0ull;
    }
    __syncthreads();
    if (s < BP_TILE) {
        for (int r = 0; r < 2; r++) {
            const uint32_t g = s_g[r][s];
            uint32_t c = 0;
            for (int k = 0; k < BP_TILE; k++) c += s_g[r][k] < g;
            s_lr[r][s] = (uint16_t)c;
        }
    }
    __syncthreads();
    // prefix tables: row r = slots of the tile whose tile-local rank is >= r  (i.e. free >= threshold)
    if (s < BP_ROWS) {
        for (int r = 0; r < 2; r++) {
            uint32_t w[8];
#pragma unroll
            for (int j = 0; j < 8; j++) {
                uint32_t acc = 0;
                for (int b = 0; b < 32; b++) {
                    const int k = j * 32 + b;
                    acc |= (uint32_t)(s_valid[k] && s_lr[r][k] >= s) << b;
                }
                w[j] = acc;
            }
            uint4* tab = reinterpret_cast<uint4*>(B + (r ? lay.off_tabM : lay.off_tabC) + table_row_offset(t, s));
            tab[0] = make_uint4(w[0], w[1], w[2], w[3]);
            tab[1] = make_uint4(w[4], w[5], w[6], w[7]);
        }
    }
    // bucket membership + base counts, layout [bucket][tile]
    unsigned long long* membC = reinterpret_cast<unsigned long long*>(B + lay.off_membC);
    unsigned long long* membM = reinterpret_cast<unsigned long long*>(B + lay.off_membM);
    uint16_t* baseC = reinterpret_cast<uint16_t*>(B + lay.off_baseC);
    uint16_t* baseM = reinterpret_cast<uint16_t*>(B + lay.off_baseM);
    for (uint32_t hi = s; hi < lay.nb; hi += blockDim.x) {
        membC[(size_t)hi * lay.nt + t] = 0ull;
        membM[(size_t)hi * lay.nt + t] = 0ull;
    }
    __syncthreads();
    if (s < BP_TILE && s_valid[s]) {
        atomicOr(&membC[(size_t)(s_g[0][s] >> 6) * lay.nt + t], 1ull << (s_g[0][s] & 63));
        atomicOr(&membM[(size_t)(s_g[1][s] >> 6) * lay.nt + t], 1ull << (s_g[1][s] & 63));
    }
    __threadfence();
    __syncthreads();
    const uint32_t warp = s >> 5, lane = s & 31;
    if (warp < 2) {
        const unsigned long long* memb = warp ? membM : membC;
        uint16_t* base = warp ? baseM : baseC;
        uint32_t running = 0;
        for (uint32_t h0 = 0; h0 < lay.nb; h0 += 32) {
            const uint32_t hi = h0 + lane;
            const uint32_t c = hi < lay.nb ? __popcll(__ldcg(&memb[(size_t)hi * lay.nt + t])) : 0;
            uint32_t inc = c;
#pragma unroll
            for (int off = 1; off < 32; off <<= 1) {
                const uint32_t o = __shfl_up_sync(0xffffffffu, inc, off);
                if (lane >= (uint32_t)off) inc += o;
            }
            if (hi < lay.nb) base[(size_t)hi * lay.nt + t] = (uint16_t)(running + inc - c);
            running += __shfl_sync(0xffffffffu, inc, 31);
        }
    }
    // label-pair columns, layout [bit][tile][8 words]
    uint8_t* pairs = B + lay.off_pairs;
    for (uint32_t bit = s; bit < 64u * nt.W; bit += blockDim.x) {
        const uint32_t w_ = bit >> 6, sh = bit & 63;
        uint32_t w[8];
#pragma unroll
        for (int j = 0; j < 8; j++) {
            uint32_t acc = 0;
            for (int b = 0; b < 32; b++) acc |= (uint32_t)((s_lab[w_][j * 32 + b] >> sh) & 1ull) << b;
            w[j] = acc;
        }
        uint4* dst = reinterpret_cast<uint4*>(pairs + (size_t)bit * lay.pstride + (size_t)t * 32);
        dst[0] = make_uint4(w[0], w[1], w[2], w[3]);
        dst[1] = make_uint4(w[4], w[5], w[6], w[7]);
    }
}

// ---- "rows" format (ks_bitpar.h): one CTA builds one 256-slot tile of a column block, node-index order ----
// Also leaves the tile's global positions in ascending order (tile_sorted) for k_build_ranks.
__global__ void __launch_bounds__(288)
    k_build_cbtile(NodeTable nt, const uint32_t* __restrict__ gposC, const uint32_t* __restrict__ gposM,
                   uint8_t* __restrict__ blob, RowsLayout lay, uint32_t* __restrict__ tile_sorted) {
    __shared__ uint32_t s_g[2][BP_TILE];
    __shared__ uint16_t s_lr[2][BP_TILE];
    __shared__ uint8_t s_valid[BP_TILE];
    __shared__ uint64_t s_lab[KS_MAX_LABEL_WORDS][BP_TILE];
    const uint32_t tile_g = blockIdx.x, cb = tile_g / RW_TILES, t = tile_g % RW_TILES, s = threadIdx.x;
    const uint32_t n_tiles_pad = lay.ncb * RW_TILES;
    uint8_t* B = blob + (size_t)cb * lay.cb_stride;
    if (s < BP_TILE) {
        const uint32_t n = tile_g * BP_TILE + s;
        const bool v = n < nt.N;
        s_valid[s] = v;
        s_g[0][s] = v ? gposC[n] : 0xFFFFFFFFu;
        s_g[1][s] = v ? gposM[n] : 0xFFFFFFFFu;
        for (uint32_t w = 0; w < nt.W; w++) s_lab[w][s] = v ? nt.labels[(size_t)w * nt.Npad + n] : 0ull;
    }
    __syncthreads();
    if (s < BP_TILE) {
        for (int r = 0; r < 2; r++) {
            const uint32_t g = s_g[r][s];
            uint32_t c = 0;
            for (int k = 0; k < BP_TILE; k++) c += s_g[r][k] < g;
            s_lr[r][s] = (uint16_t)c;
            // positions are distinct, so the valid slots fill tile_sorted[0..count) exactly; the rest is +inf
            uint32_t* ts = tile_sorted + ((size_t)r * n_tiles_pad + tile_g) * BP_TILE;
            if (s_valid[s]) ts[c] = g;
            const uint32_t count = nt.N > tile_g * BP_TILE ? min((uint32_t)BP_TILE, nt.N - tile_g * BP_TILE) : 0u;
            if (s >= count) ts[s] = 0xFFFFFFFFu;
        }
    }
    __syncthreads();
    // prefix tables: row r = slots of the tile whose tile-local rank is >= r  (i.e. free >= threshold)
    if (s < BP_ROWS) {
        for (int r = 0; r < 2; r++) {
            uint32_t w[8];
#pragma unroll
            for (int j = 0; j < 8; j++) {
                uint32_t acc = 0;
                for (int b = 0; b < 32; b++) {
                    const int k = j * 32 + b;
                    acc |= (uint32_t)(s_valid[k] && s_lr[r][k] >= s) << b;
                }
                w[j] = acc;
            }
            uint8_t* line = B + (r ? lay.off_tabM : lay.off_tabC) + (size_t)s * RW_LINE + t * 16;
            *reinterpret_cast<uint4*>(line) = make_uint4(w[0], w[1], w[2], w[3]);
            *reinterpret_cast<uint4*>(line + 128) = make_uint4(w[4], w[5], w[6], w[7]);
        }
    }
    // label-pair columns
    for (uint32_t bit = s; bit < 64u * nt.W; bit += blockDim.x) {
        const uint32_t w_ = bit >> 6, sh = bit & 63;
        uint32_t w[8];
#pragma unroll
        for (int j = 0; j < 8; j++) {
            uint32_t acc = 0;
            for (int b = 0; b < 32; b++) acc |= (uint32_t)((s_lab[w_][j * 32 + b] >> sh) & 1ull) << b;
            w[j] = acc;
        }
        uint8_t* line = B + lay.off_pairs + (size_t)bit * RW_LINE + t * 16;
        *reinterpret_cast<uint4*>(line) = make_uint4(w[0], w[1], w[2], w[3]);
        *reinterpret_cast<uint4*>(line + 128) = make_uint4(w[4], w[5], w[6], w[7]);
    }
}

// rank tables: rank[cb][g][resource][t] = number of nodes of tile (cb, t) at sorted positions < g in that
// resource's order, for every threshold g in [0, N].  One thread = one threshold of one column block: 8 binary searches per resource over the tile's
// sorted positions (shared memory), one 16-byte store per resource.
__global__ void __launch_bounds__(256)
    k_build_ranks(const uint32_t* __restrict__ tile_sorted, RowsLayout lay, uint16_t* __restrict__ rank) {
    __shared__ uint32_t s_pos[2][RW_TILES][BP_TILE];
    const uint32_t cb = blockIdx.y, n_tiles_pad = lay.ncb * RW_TILES;
    for (uint32_t i = threadIdx.x; i < 2 * RW_TILES * BP_TILE; i += blockDim.x) {
        const uint32_t r = i / (RW_TILES * BP_TILE), tt = (i / BP_TILE) % RW_TILES, k = i % BP_TILE;
        s_pos[r][tt][k] = tile_sorted[((size_t)r * n_tiles_pad + cb * RW_TILES + tt) * BP_TILE + k];
    }
    __syncthreads();
    const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= lay.n_thr) return;
#pragma unroll
    for (int r = 0; r < 2; r++) {
        uint32_t out[RW_TILES];
#pragma unroll
        for (uint32_t tt = 0; tt < RW_TILES; tt++) {
            const uint32_t* a = s_pos[r][tt];
            uint32_t lo = 0; // number of elements < g (0..256)
#pragma unroll
            for (uint32_t step = BP_TILE / 2; step > 0; step >>= 1)
                if (a[lo + step - 1] < g) lo += step;
            if (a[lo] < g) lo++; // lo <= 255 here
            out[tt] = lo;
        }
        uint16_t* dst = rank + (((size_t)cb * lay.n_thr + g) * 2 + r) * RW_TILES; // [cb][g][resource][tile]
        *reinterpret_cast<uint4*>(dst) = make_uint4(out[0] | (out[1] << 16), out[2] | (out[3] << 16),
                                                   out[4] | (out[5] << 16), out[6] | (out[7] << 16));
    }
}

// ------------------------------------------------------------------------------------------------ per call
template <class Ptr>
__device__ __forceinline__ uint32_t lower_bound_i64(Ptr a, uint32_t n, int64_t x) {
    uint32_t lo = 0, len = n; // number of elements < x
    while (len > 0) {
        const uint32_t half = len >> 1;
        if (a[lo + half] < x) {
            lo += half + 1;
            len -= half + 1;
        } else {
            len = half;
        }
    }
    return lo;
}

// rank = number of nodes with free < request; nodes at sorted positions >= rank satisfy request <= free
// (predicates.rs:42).  Two-level search: <=2048 splitters per resource in shared memory, then a window of
// spl_stride-1 elements of the global sorted array.
// The same kernel writes the mask kernel's pod records (thresholds, pod index, selector columns) in pod order: round 1
// sorted the pods by threshold to tame shared-memory bank conflicts; the rows format is conflict-free for any order and
// measured faster without the sort (profiles/r02_experiments.txt).
constexpr uint32_t RW_SEL_GENERIC = 0xFFFFFFFFu;
constexpr uint32_t RW_PID_NONE = 0xFFFFFFFFu;

// the selector of a pod as record word: up to three required label-pair bit indices (10 bits each) + their number in
// bits 30-31; RW_SEL_GENERIC when it names more than three pairs (the mask kernel then walks the selector words)
template <class LoadWord>
__device__ __forceinline__ uint32_t selector_record(uint32_t W, LoadWord word) {
    uint32_t cols = 0, n_req = 0;
    for (uint32_t w = 0; w < W; w++) {
        unsigned long long bits = word(w);
        while (bits) { // required (key,value) pairs of the selector (predicates.rs:48)
            const uint32_t bit = w * 64 + __ffsll((long long)bits) - 1;
            bits &= bits - 1;
            if (n_req < 3) cols |= bit << (10 * n_req);
            n_req++;
        }
    }
    return n_req > 3 ? RW_SEL_GENERIC : (cols | (n_req << 30));
}

__global__ void __launch_bounds__(RANK_THREADS, 1)
    k_pod_ranks(PodView pv, const int64_t* __restrict__ sortedC, const int64_t* __restrict__ sortedM, uint32_t N,
                const int64_t* __restrict__ splC, const int64_t* __restrict__ splM, uint32_t n_spl, uint32_t stride,
                uint2* __restrict__ rk, uint32_t* __restrict__ cnt_zero, uint32_t W, uint4* __restrict__ rec,
                uint32_t* __restrict__ cursor, uint32_t n_cursor) {
    extern __shared__ __align__(16) unsigned char ranks_smem[];
    int64_t* const s_spl[2] = {reinterpret_cast<int64_t*>(ranks_smem), reinterpret_cast<int64_t*>(ranks_smem) + n_spl};
    if (threadIdx.x == 0) trace_start(TR_RANKS_START);
    if (blockIdx.x == 0) // the mask kernel's chunk cursors
        for (uint32_t k = threadIdx.x; k < n_cursor; k += blockDim.x) cursor[(size_t)k * RW_CURSOR_STRIDE] = 0;
    for (uint32_t k = threadIdx.x; k < n_spl; k += blockDim.x) {
        s_spl[0][k] = splC[k];
        s_spl[1][k] = splM[k];
    }
    __syncthreads();
    if (rec) // padding of the last group of 8
        for (uint32_t p = pv.P + blockIdx.x * blockDim.x + threadIdx.x; p < ((pv.P + 7u) & ~7u); p += gridDim.x * blockDim.x)
            rec[p] = make_uint4(0, 0, RW_PID_NONE, 0);
    // Two pods per thread and pass, i.e. four searches (2 pods x 2 resources) side by side: the part over the sorted array
    // in global memory is a chain of dependent L2 loads, and the four chains advance in lockstep (4 loads in flight).
    const uint32_t T = gridDim.x * blockDim.x;
    for (uint32_t p0 = blockIdx.x * blockDim.x + threadIdx.x; p0 < pv.P; p0 += 2 * T) {
        int64_t x[4];
        uint32_t lo[4], len[4];
#pragma unroll
        for (int k = 0; k < 4; k++) { // k = 2 * pod + resource; a missing second pod searches for "below everything": no probes
            const uint32_t p = p0 + (k >> 1) * T;
            x[k] = p >= pv.P ? INT64_MIN : (k & 1) ? __ldg(pv.req_mem + p) : __ldg(pv.req_cpu + p);
        }
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const uint32_t c = lower_bound_i64(s_spl[k & 1], n_spl, x[k]);
            lo[k] = c > 0 ? (c - 1) * stride + 1 : 0u; // sorted[lo-1] < x <= sorted[c*stride] (if it exists)
            len[k] = c > 0 ? min(stride - 1, N - lo[k]) : 0u;
        }
        while (len[0] | len[1] | len[2] | len[3]) {
            int64_t v[4];
#pragma unroll
            for (int k = 0; k < 4; k++) {
                const int64_t* sorted = (k & 1) ? sortedM : sortedC;
                v[k] = len[k] ? __ldg(sorted + lo[k] + (len[k] >> 1)) : 0;
            }
#pragma unroll
            for (int k = 0; k < 4; k++) {
                const uint32_t half = len[k] >> 1;
                if (len[k] == 0) continue;
                if (v[k] < x[k]) {
                    lo[k] += half + 1;
                    len[k] -= half + 1;
                } else {
                    len[k] = half;
                }
            }
        }
#pragma unroll
        for (int q = 0; q < 2; q++) {
            const uint32_t p = p0 + q * T;
            if (p >= pv.P) break;
            rk[p] = make_uint2(lo[2 * q], lo[2 * q + 1]);
            if (cnt_zero) cnt_zero[p] = 0; // k_mask_rows accumulates feasible counts with REDs
            if (rec) // the mask kernel's 16-byte pod record, in pod order
                rec[p] = make_uint4(lo[2 * q], lo[2 * q + 1], p,
                                    selector_record(W, [&](uint32_t w) { return __ldg(pv.sel + (size_t)p * W + w); }));
        }
    }
    if (c_trace) {
        __syncthreads();
        if (threadIdx.x == 0) trace_end(TR_RANKS_END);
    }
}

// ------------------------------------------------------------------------------------------------ rows kernel
// k_mask_rows: the round-2 mask / count kernel ("rows" format, ks_bitpar.h).
//   * lane = (pod slot, tile): 8 lanes per pod = the 8 tiles of the column block = 256 contiguous bytes of the
//     pod's mask row per 256-bit store; a warp iteration covers 8 consecutive pods (two per thread, two
//     independent dependency chains);
//   * the tile-local rank of the pod's thresholds comes from the rank tables (one 16-bit load per resource from
//     L1/L2; the 8 lanes of a pod read 16 contiguous bytes) - no base/membership lookup, no POPC for ranks;
//   * table rows and label-pair columns are octet-interleaved: the 8 lanes of a shared-memory phase read granule t
//     of their own 256-byte line -> conflict-free for any ranks, plain (unswapped) stores;
//   * work = (column block, pod group) items handed out dynamically: one atomic cursor per column block, warps claim
//     RW_CLAIM groups at a time, a CTA whose block is exhausted re-stages the blob of the block with the most work left
//     (all SMs busy whatever ncb is, and SMs that stream faster simply claim more);
//   * pod records (pod order: no sort) are fetched one iteration ahead.
__device__ __forceinline__ uint4 lds128(uint32_t a) { // pure: scheduled freely; ordered after the blob wait by the
    uint4 v;                                          // address dependence on the post-wait token
    asm("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a));
    return v;
}
__device__ __forceinline__ uint32_t ldg_u16_keep(const uint16_t* p, uint64_t pol) { // L2 evict-last: the rank tables are re-read
    uint32_t v;
    asm("ld.global.nc.L2::cache_hint.u16 %0, [%1], %2;" : "=r"(v) : "l"(p), "l"(pol));
    return v;
}
template <class T>
__device__ __forceinline__ T* opaque_ptr(T* p) { // keeps a per-thread base pointer in one register pair (the compiler
    asm("" : "+l"(p));                           // would otherwise re-derive its lane part in every iteration)
    return p;
}
__device__ __forceinline__ uint4 and4(uint4 a, uint4 b) { return make_uint4(a.x & b.x, a.y & b.y, a.z & b.z, a.w & b.w); }
__device__ __forceinline__ uint4 and4(uint4 a, uint4 b, uint4 c) {
    return make_uint4(a.x & b.x & c.x, a.y & b.y & c.y, a.z & b.z & c.z, a.w & b.w & c.w);
}
struct RowsParams { // kernel parameters stay in the constant bank: the loop reads them from there on demand
    const uint8_t* blob;
    RowsLayout lay;
    const uint16_t* rank;            // [cb][threshold g][resource][tile] u16: 32 bytes per (cb, g)
    const uint4* rec_s;              // sorted pod records, padded to a multiple of 8
    const unsigned long long* sel_s; // the pods' selector words, pod order (generic path only)
    uint32_t n_groups;               // groups of 8 pods
    uint32_t* mask;                  // may be nullptr
    uint32_t row_words;              // mask row pitch in 32-bit words
    uint32_t* cnt;                   // may be nullptr
    uint32_t* cursor;                // [ncb * RW_CURSOR_STRIDE] next unclaimed pod group of every column block
};
constexpr uint32_t RW_CLAIM = 4;     // pod groups per claim (one atomicAdd per warp and ~4 x 2 KB x 8 of mask)
constexpr uint32_t RW_HOP_MIN = 256; // a partly claimed column block is worth moving to while it has this many groups left

// one (pod, tile) item: 256 cells -> mask words a (0..3), b (4..7); returns the number of feasible cells.
// a_tab = shared-window address of granule t of line 0 of tabC; tabM and the pair columns sit at constant offsets.
template <int W, bool PSMEM>
__device__ __forceinline__ uint32_t rows_item(const RowsParams& prm, uint32_t a_tab, uint32_t cb, uint32_t t, uint32_t* mask_col,
                                              uint32_t rC, uint32_t rM, uint32_t pid, uint32_t sel, uint32_t q, uint64_t pol_st) {
    const uint32_t aC = a_tab + rC * RW_LINE, aM = a_tab + rM * RW_LINE;
    const uint4 c0 = lds128(aC), c1 = lds128(aC + 128);
    const uint4 m0 = lds128(aM + RW_TAB_BYTES), m1 = lds128(aM + RW_TAB_BYTES + 128);
    uint4 a, b;
    auto column = [&](uint32_t bit, uint4& q0, uint4& q1) { // node column of one required pair (predicates.rs:48-53)
        if (PSMEM) {
            const uint32_t ap = a_tab + bit * RW_LINE;
            q0 = lds128(ap + 2 * RW_TAB_BYTES);
            q1 = lds128(ap + 2 * RW_TAB_BYTES + 128);
        } else {
            const uint4* gp = reinterpret_cast<const uint4*>(prm.blob + (size_t)cb * prm.lay.cb_stride + prm.lay.off_pairs +
                                                             (size_t)bit * RW_LINE + t * 16u);
            q0 = __ldg(gp);
            q1 = __ldg(gp + 8);
        }
    };
    const uint32_t n_req = sel >> 30;
    if (n_req == 0) {
        a = and4(c0, m0);
        b = and4(c1, m1);
    } else if (sel != RW_SEL_GENERIC) {
        uint4 q0, q1;
        column(sel & 0x3FFu, q0, q1);
        a = and4(c0, m0, q0);
        b = and4(c1, m1, q1);
        if (n_req >= 2) {
            column((sel >> 10) & 0x3FFu, q0, q1);
            a = and4(a, q0);
            b = and4(b, q1);
            if (n_req == 3) {
                column((sel >> 20) & 0x3FFu, q0, q1);
                a = and4(a, q0);
                b = and4(b, q1);
            }
        }
    } else { // rare: more than three required pairs
        a = and4(c0, m0);
        b = and4(c1, m1);
#pragma unroll
        for (int w = 0; w < W; w++) {
            unsigned long long bits = __ldg(prm.sel_s + (size_t)q * W + w);
            while (bits) {
                const uint32_t bit = w * 64 + __ffsll((long long)bits) - 1;
                bits &= bits - 1;
                uint4 q0, q1;
                column(bit, q0, q1);
                a = and4(a, q0);
                b = and4(b, q1);
            }
        }
    }
    if (mask_col != nullptr && pid != RW_PID_NONE) {
        uint32_t* dst = mask_col + (size_t)pid * prm.row_words; // 32-byte aligned
        // the mask is write-once streaming data: first in line for eviction from L2 (plain stores: +2.4 % kernel time)
        asm volatile("st.global.L2::cache_hint.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8}, %9;" ::"l"(dst), "r"(a.x), "r"(a.y),
                     "r"(a.z), "r"(a.w), "r"(b.x), "r"(b.y), "r"(b.z), "r"(b.w), "l"(pol_st)
                     : "memory");
    }
    return __popc(a.x) + __popc(a.y) + __popc(a.z) + __popc(a.w) + __popc(b.x) + __popc(b.y) + __popc(b.z) + __popc(b.w);
}

// (launch bounds of 1024 threads for both block sizes: 64 registers per thread, so that a 768-thread CTA leaves a quarter
// of the register file to the argmax CTAs that run beside it)
template <int W, bool PSMEM, int THREADS>
__global__ void __launch_bounds__(BP_THREADS, 1) k_mask_rows(const __grid_constant__ RowsParams prm) {
    extern __shared__ __align__(128) uint8_t smem[];
    __shared__ __align__(8) uint64_t bar;
    __shared__ unsigned long long s_key;
    const uint32_t tid = threadIdx.x, t = tid & 7, ps = (tid >> 3) & 3;
    uint64_t pol_st, pol_ld; // L2 policies: mask stores evict-first, rank-table loads evict-last
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol_st));
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol_ld));
    if (tid == 0) {
        mbar_init(&bar, 1);
        fence_mbar_init();
        trace_start(TR_MASK_START);
    }
    __syncthreads();
    uint32_t phase = 0;

    // Work = (column block, pod group) items.  Every column block has one cursor (zeroed by k_pod_ranks); a warp claims
    // RW_CLAIM consecutive pod groups of the staged column block at a time with one atomicAdd, one claim ahead of the one
    // it is working on.  The CTAs that share a column block therefore finish it together whatever their individual rates
    // (with equal static shares the first CTA finished 11 % before the last one on C3: SMs do not all stream at the same
    // rate), and a CTA whose block is exhausted moves - one barrier, one re-staging of the 148 KB blob - to the block
    // with the most unclaimed groups.  CTAs start spread evenly over the column blocks.
    const uint32_t n_slots = prm.n_groups; // pod groups per column block
    const uint32_t ncb = prm.lay.ncb;
    const uint32_t lane = tid & 31;
    const uint32_t last_grp = n_slots - 1;
    const uint4* rec_t = opaque_ptr(prm.rec_s + 2 * ps); // this thread's pods: 2*ps and 2*ps+1 of the group (neighbours)
    // loads are unconditional (group index clamped into the list)
    auto fetch_rec = [&](uint32_t j, uint4& ra, uint4& rb) {
        const uint4* rp = rec_t + (size_t)min(j, last_grp) * 8u;
        ra = __ldg(rp);
        rb = __ldg(rp + 1);
    };
    uint32_t cb = (uint32_t)((uint64_t)blockIdx.x * ncb / gridDim.x);
    for (;;) { // one iteration per column block this CTA works on
        __syncthreads(); // all reads of the previous blob are done
        if (tid == 0) {
            fence_proxy_async();
            mbar_arrive_expect_tx(&bar, prm.lay.smem_bytes);
            const uint8_t* src = prm.blob + (size_t)cb * prm.lay.cb_stride;
            for (uint32_t off = 0; off < prm.lay.smem_bytes; off += 32768u)
                tma_bulk_g2s(smem + off, src + off, min(32768u, prm.lay.smem_bytes - off), &bar);
        }
        uint32_t* cursor = prm.cursor + (size_t)cb * RW_CURSOR_STRIDE;
        auto claim = [&]() -> uint32_t { // lane 0 holds the result; broadcast where it is needed
            return lane == 0 ? atomicAdd(cursor, RW_CLAIM) : 0u;
        };
        uint32_t base = __shfl_sync(0xffffffffu, claim(), 0);
        uint32_t next_raw = claim();
        // rank entry of (g, resource r, tile t): rk_t[g * 16 + r * 8]
        const uint16_t* rk_t = opaque_ptr(prm.rank + (size_t)cb * prm.lay.n_thr * (2 * RW_TILES) + t);
        auto fetch_ranks = [&](const uint4& ra, const uint4& rb, uint32_t& rCa, uint32_t& rMa, uint32_t& rCb, uint32_t& rMb) {
            rCa = ldg_u16_keep(rk_t + (size_t)ra.x * 16u, pol_ld);
            rMa = ldg_u16_keep(rk_t + (size_t)ra.y * 16u + 8, pol_ld);
            rCb = ldg_u16_keep(rk_t + (size_t)rb.x * 16u, pol_ld);
            rMb = ldg_u16_keep(rk_t + (size_t)rb.y * 16u + 8, pol_ld);
        };
        // records of iteration k+1 are in flight while k computes (its ranks are loaded at the top of k; a deeper pipeline
        // - records two ahead, ranks one ahead - measured 2 % slower: profiles/r02_experiments.txt)
        uint4 nA, nB;
        fetch_rec(base, nA, nB);

        mbar_wait(&bar, phase);
        phase ^= 1;
        uint32_t tok; // every shared-memory load below depends on a value produced after the wait
        asm volatile("mov.u32 %0, 0;" : "=r"(tok)::"memory");
        const uint32_t a_tab = smem_u32(smem) + t * 16u + tok;
        const uint32_t tile = cb * RW_TILES + t;
        // a tile is written when it holds nodes, or when the caller's row pitch has room for it (a pitch that is a multiple
        // of 256 bytes - ks_mask_row_bytes_aligned - lets the 8 lanes of a pod always store one whole, 256-byte-aligned
        // block: partial blocks cost a third of the store bandwidth, profiles/r02_write_bw_v2.txt); padding tiles hold zeros
        uint32_t* mask_col = (prm.mask != nullptr && (tile < prm.lay.n_tiles || (tile + 1u) * 8u <= prm.row_words))
                                 ? opaque_ptr(prm.mask + (size_t)tile * 8u)
                                 : nullptr;

        while (base < n_slots) { // warp-uniform: one claim of up to RW_CLAIM pod groups
            const uint32_t end = min(base + RW_CLAIM, n_slots);
            uint32_t next = 0;
            for (uint32_t j = base; j < end; j++) {
                const uint32_t pidA = nA.z, selA = nA.w, pidB = nB.z, selB = nB.w;
                uint32_t rCa, rMa, rCb, rMb;
                fetch_ranks(nA, nB, rCa, rMa, rCb, rMb);
                uint32_t jn = j + 1;
                if (jn == end) { // last group of the claim: the next claim (requested a whole claim ago) says what follows
                    next = __shfl_sync(0xffffffffu, next_raw, 0);
                    jn = next;
                }
                fetch_rec(jn, nA, nB);
                const uint32_t cA = rows_item<W, PSMEM>(prm, a_tab, cb, t, mask_col, rCa, rMa, pidA, selA, j * 8u + 2u * ps, pol_st);
                const uint32_t cB = rows_item<W, PSMEM>(prm, a_tab, cb, t, mask_col, rCb, rMb, pidB, selB, j * 8u + 2u * ps + 1u, pol_st);
                if (prm.cnt != nullptr) { // the 8 lanes of a pod are adjacent; both pods' counts ride in one register
                    uint32_t c = cA | (cB << 16);
                    c += __shfl_xor_sync(0xffffffffu, c, 1);
                    c += __shfl_xor_sync(0xffffffffu, c, 2);
                    c += __shfl_xor_sync(0xffffffffu, c, 4);
                    if (t == 0) {
                        const uint32_t ca = c & 0xFFFFu, cb_ = c >> 16;
                        if (ncb == 1) { // single writer, no zero-init needed
                            if (pidA != RW_PID_NONE) prm.cnt[pidA] = ca;
                            if (pidB != RW_PID_NONE) prm.cnt[pidB] = cb_;
                        } else {
                            if (pidA != RW_PID_NONE && ca) atomicAdd(&prm.cnt[pidA], ca);
                            if (pidB != RW_PID_NONE && cb_) atomicAdd(&prm.cnt[pidB], cb_);
                        }
                    }
                }
            }
            base = next;
            if (base < n_slots) next_raw = claim();
        }

        // this column block is exhausted (its last groups are being finished by the warps that claimed them, here or in
        // other CTAs): move to the block with the most unclaimed groups, if any is worth a re-staging
        if (ncb == 1) break;
        __syncthreads();
        if (tid == 0) s_key = 0;
        __syncthreads();
        for (uint32_t c = tid; c < ncb; c += THREADS) {
            const uint32_t used = *reinterpret_cast<volatile uint32_t*>(prm.cursor + (size_t)c * RW_CURSOR_STRIDE);
            const uint32_t left = used < n_slots ? n_slots - used : 0u;
            if (left >= RW_HOP_MIN || (left > 0 && used == 0)) { // key: groups left, then nearness to the current block
                const uint32_t dist = (c + ncb - cb) % ncb;
                atomicMax(&s_key, ((unsigned long long)left << 32) | (0xFFFFFFFFu - dist));
            }
        }
        __syncthreads();
        const unsigned long long key = s_key;
        if (key == 0) break;
        cb = (cb + (0xFFFFFFFFu - (uint32_t)key)) % ncb;
    }
    if (c_trace) {
        __syncthreads();
        if (tid == 0) {
            const unsigned long long now = global_ns();
            atomicMax(c_trace + TR_MASK_END, now);
            atomicMax(c_trace + TR_MASK_FIRST_CTA_END_INV, ~now); // = ~(earliest CTA end)
        }
    }
}

// ---- argmax of the separable score = first feasible node in descending priority order ----
// The priority-ordered index (blobP) is read through L1/L2.  Phase 1 (k_first_fit_head): one thread per pod
// looks at the two best tiles (512 best nodes) - enough for almost every pod; the rest is appended to a list.
// Phase 2 (k_first_fit_tail): one warp per listed pod, one tile per lane, 32 tiles per step, ballot + early exit.
struct PodThreshold {
    const uint16_t* baseC;
    const uint16_t* baseM;
    const unsigned long long* membC;
    const unsigned long long* membM;
    unsigned long long lowC, lowM;
};

__device__ __forceinline__ PodThreshold pod_threshold(const uint8_t* __restrict__ blobP, const BitparLayout& lay, uint2 r) {
    PodThreshold t;
    t.baseC = reinterpret_cast<const uint16_t*>(blobP + lay.off_baseC) + (size_t)(r.x >> 6) * lay.nt;
    t.baseM = reinterpret_cast<const uint16_t*>(blobP + lay.off_baseM) + (size_t)(r.y >> 6) * lay.nt;
    t.membC = reinterpret_cast<const unsigned long long*>(blobP + lay.off_membC) + (size_t)(r.x >> 6) * lay.nt;
    t.membM = reinterpret_cast<const unsigned long long*>(blobP + lay.off_membM) + (size_t)(r.y >> 6) * lay.nt;
    t.lowC = (1ull << (r.x & 63)) - 1ull;
    t.lowM = (1ull << (r.y & 63)) - 1ull;
    return t;
}

template <int W>
__device__ __forceinline__ void ptile_mask(const uint8_t* __restrict__ blobP, const BitparLayout& lay, const PodThreshold& t,
                                           const unsigned long long (&sel)[W], uint32_t k, uint32_t (&m)[8]) {
    const uint32_t rankC = __ldg(t.baseC + k) + __popcll(__ldg(t.membC + k) & t.lowC);
    const uint32_t rankM = __ldg(t.baseM + k) + __popcll(__ldg(t.membM + k) & t.lowM);
    const uint4* tc = reinterpret_cast<const uint4*>(blobP + lay.off_tabC + table_row_offset(k, rankC));
    const uint4* tm = reinterpret_cast<const uint4*>(blobP + lay.off_tabM + table_row_offset(k, rankM));
    const uint4 c0 = __ldg(tc), c1 = __ldg(tc + 1);
    const uint4 m0 = __ldg(tm), m1 = __ldg(tm + 1);
    m[0] = c0.x & m0.x; m[1] = c0.y & m0.y; m[2] = c0.z & m0.z; m[3] = c0.w & m0.w;
    m[4] = c1.x & m1.x; m[5] = c1.y & m1.y; m[6] = c1.z & m1.z; m[7] = c1.w & m1.w;
    const uint8_t* pairs = blobP + lay.off_pairs;
#pragma unroll
    for (int w = 0; w < W; w++) {
        unsigned long long bits = sel[w];
        while (bits) {
            const uint32_t bit = w * 64 + __ffsll((long long)bits) - 1;
            bits &= bits - 1;
            const uint4* col = reinterpret_cast<const uint4*>(pairs + (size_t)bit * lay.pstride + (size_t)k * 32);
            const uint4 q0 = __ldg(col);
            const uint4 q1 = __ldg(col + 1);
            m[0] &= q0.x; m[1] &= q0.y; m[2] &= q0.z; m[3] &= q0.w;
            m[4] &= q1.x; m[5] &= q1.y; m[6] &= q1.z; m[7] &= q1.w;
        }
    }
}

__device__ __forceinline__ int first_bit_256(const uint32_t (&m)[8]) {
    int first = -1;
#pragma unroll
    for (int j = 7; j >= 0; j--)
        if (m[j]) first = j * 32 + __ffs(m[j]) - 1;
    return first;
}

__device__ __forceinline__ void write_binding(const OutView& ov, const PodView& pv, const PeerOut& po, uint32_t p, int slot,
                                              const int32_t* __restrict__ ord_idx, const int64_t* __restrict__ ord_prio) {
    int32_t best = -1;
    int64_t score = 0;
    if (slot >= 0) {
        best = __ldg(ord_idx + slot);
        score = __ldg(ord_prio + slot) - leftover_cost(__ldg(pv.req_cpu + p), __ldg(pv.req_mem + p));
    }
    store_binding(ov, po, p, best, score);
}

constexpr uint32_t FF_HEAD_TILES = 2;

template <int W>
__global__ void __launch_bounds__(256)
    k_first_fit_head(const uint8_t* __restrict__ blobP, BitparLayout lay, const int32_t* __restrict__ ord_idx,
                     const int64_t* __restrict__ ord_prio, PodView pv, const uint2* __restrict__ rk, OutView ov,
                     uint32_t* __restrict__ tail_list, uint32_t* __restrict__ tail_count, PeerOut po, bool last_kernel,
                     const unsigned long long* __restrict__ live, uint32_t N) {
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p == 0) exchange_stamp(po, 0);
    if (threadIdx.x == 0) trace_start(TR_ARGMAX1_START);
    if (p < pv.P) {
        const uint2 r = __ldg(rk + p);
        const PodThreshold t = pod_threshold(blobP, lay, r);
        unsigned long long sel[W];
        bool dead = r.x >= N || r.y >= N; // the request exceeds every node's free cpu / memory
#pragma unroll
        for (int w = 0; w < W; w++) {
            sel[w] = __ldg(pv.sel + (size_t)p * W + w);
            dead |= (sel[w] & ~__ldg(live + w)) != 0; // a required pair that no node carries
        }
        if (dead) { // infeasible everywhere: answered without scanning the 196 tiles in the tail kernel
            write_binding(ov, pv, po, p, -1, ord_idx, ord_prio);
        } else {
        uint32_t m0[8], m1[8];
        ptile_mask<W>(blobP, lay, t, sel, 0, m0);
        ptile_mask<W>(blobP, lay, t, sel, min(1u, lay.nt - 1), m1);
        int slot = first_bit_256(m0);
        if (slot < 0 && lay.nt > 1) {
            const int s1 = first_bit_256(m1);
            if (s1 >= 0) slot = BP_TILE + s1;
        }
        if (slot >= 0 || lay.nt <= FF_HEAD_TILES) write_binding(ov, pv, po, p, slot, ord_idx, ord_prio);
        else tail_list[atomicAdd(tail_count, 1u)] = p; // order of the list does not affect any result
        }
    }
    if (c_trace) {
        __syncthreads();
        if (threadIdx.x == 0) trace_end(TR_ARGMAX1_END);
    }
    if (last_kernel) exchange_signal(po); // no tail kernel follows: this rank's bindings are complete
}

template <int W>
__global__ void __launch_bounds__(256)
    k_first_fit_tail(const uint8_t* __restrict__ blobP, BitparLayout lay, const int32_t* __restrict__ ord_idx,
                     const int64_t* __restrict__ ord_prio, PodView pv, const uint2* __restrict__ rk, OutView ov,
                     const uint32_t* __restrict__ tail_list, const uint32_t* __restrict__ tail_count, PeerOut po) {
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t warps = gridDim.x * (blockDim.x >> 5);
    const uint32_t n = *tail_count;
    if (blockIdx.x == 0 && threadIdx.x == 0) exchange_stamp(po, 4);
    if (threadIdx.x == 0) trace_start(TR_ARGMAX2_START);
    for (uint32_t i = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); i < n; i += warps) {
        const uint32_t p = tail_list[i];
        const PodThreshold t = pod_threshold(blobP, lay, __ldg(rk + p));
        unsigned long long sel[W];
#pragma unroll
        for (int w = 0; w < W; w++) sel[w] = __ldg(pv.sel + (size_t)p * W + w);
        int slot = -1;
        for (uint32_t k0 = FF_HEAD_TILES; k0 < lay.nt; k0 += 32) {
            const uint32_t k = k0 + lane;
            int s = -1;
            if (k < lay.nt) {
                uint32_t m[8];
                ptile_mask<W>(blobP, lay, t, sel, k, m);
                s = first_bit_256(m);
            }
            const uint32_t b = __ballot_sync(0xffffffffu, s >= 0);
            if (b) { // lowest tile index = highest priority
                const int src = __ffs(b) - 1;
                slot = (int)((k0 + src) * BP_TILE) + __shfl_sync(0xffffffffu, s, src);
                break;
            }
        }
        if (lane == 0) write_binding(ov, pv, po, p, slot, ord_idx, ord_prio);
    }
    if (c_trace) {
        __syncthreads();
        if (threadIdx.x == 0) trace_end(TR_ARGMAX2_END);
    }
    exchange_signal(po); // the head kernel's stores completed before this kernel started
}

// ---- argmax of KS_SCORE_LEAST_ALLOCATED (not separable): bound-ordered scan with early exit ----
// Nodes are visited in descending order of least_alloc_bound (ties by node index), 256 at a time through the same
// table machinery (blobL); every feasible node of a tile is scored exactly; the scan stops as soon as the best exact
// score beats the bound of everything that follows.  One warp per pod: all lanes derive the tile's feasibility mask,
// lane l scores the set bits of word l&7 whose position is congruent to l>>3 mod 4; shuffle argmax per tile.
// Pods with a negative request (allowed by the ABI, never produced by a Kubernetes object) void the bound: they scan
// every tile, which is still exact.
struct NodeEval { // one row per slot of the bound order
    int64_t fc, fm, ac, am;
    double inv_ac, inv_am; // 1/alloc: quotient estimate, corrected to the exact floor below
    int32_t idx;
    int32_t pad;
};

// Single-precision view of the same row: in the common case it gives k_least_alloc the EXACT integer score of a cell
// without the 64-byte row and the two 64-bit divisions.  x = (float)free_cpu and y = (float)alloc_cpu when they are
// exactly representable (|free_cpu| < 2^24, 0 < alloc_cpu < 2^24; y = +inf for alloc_cpu <= 0, where the cpu term is 0
// by definition; NaN otherwise): for a request that is exact too, t = (x - r) * 100 is exact while t < 2^24, and the
// floor of the correctly rounded quotient t / y of two such integers IS floor((free_cpu - r) * 100 / alloc_cpu) (a
// quotient that is not an integer is at least 1 / y away from one, more than the rounding error t / y * 2^-24 for
// t < 2^24).  Memory is in bytes and does not fit: z = free_mem * 100 / alloc_mem and w = 100 / alloc_mem (both 0 for
// alloc_mem <= 0) give the real-valued quotient z - r * w with a relative error of a few 2^-24; its floor is known
// whenever no integer lies within the error bound (the kernel uses 2e-6 * (|z| + |r * w|) + 1e-3, > 8 x the worst case).
__global__ void __launch_bounds__(256)
    k_build_eval(NodeTable nt, const int32_t* __restrict__ ordL_idx, uint32_t Nord, NodeEval* __restrict__ ev,
                 float4* __restrict__ hint) {
    const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= Nord) return;
    const int32_t n = ordL_idx[s];
    NodeEval e;
    e.idx = n;
    e.pad = 0;
    if (n >= 0) {
        e.fc = nt.free_cpu[n];
        e.fm = nt.free_mem[n];
        e.ac = nt.alloc_cpu[n];
        e.am = nt.alloc_mem[n];
    } else {
        e.fc = e.fm = INT64_MIN;
        e.ac = e.am = 0;
    }
    e.inv_ac = e.ac > 0 ? 1.0 / (double)e.ac : 0.0;
    e.inv_am = e.am > 0 ? 1.0 / (double)e.am : 0.0;
    ev[s] = e;
    const float qnan = __int_as_float(0x7fc00000);
    const bool fc_exact = e.fc > -(1ll << 24) && e.fc < (1ll << 24);
    const double Sm = e.am > 0 ? (double)e.fm * 100.0 * e.inv_am : 0.0;
    hint[s] = make_float4(fc_exact ? (float)e.fc : qnan, e.ac <= 0 ? INFINITY : (e.ac < (1ll << 24) ? (float)e.ac : qnan), (float)Sm,
                          (float)(100.0 * e.inv_am));
}

// floor(x / d) for x >= 0, d > 0 (both < 2^63): double estimate, then exact correction in integers
__device__ __forceinline__ int64_t div_floor_pos(int64_t x, int64_t d, double inv_d) {
    int64_t q = (int64_t)((double)x * inv_d);
    int64_t r = x - q * d;
    while (r < 0) {
        q--;
        r += d;
    }
    while (r >= d) {
        q++;
        r -= d;
    }
    return q;
}

// the same value as least_alloc_score(e.fc, e.fm, e.ac, e.am, rc, rm) (ks_internal.cuh), with the division by a
// reciprocal (x may be negative only when the request is negative, where the generic operator is used)
__device__ __forceinline__ int64_t least_alloc_score(const NodeEval& e, int64_t rc, int64_t rm) {
    int64_t pc = 0, pm = 0;
    if (e.ac > 0) {
        const int64_t x = (e.fc - rc) * 100;
        pc = x >= 0 ? div_floor_pos(x, e.ac, e.inv_ac) : x / e.ac;
    }
    if (e.am > 0) {
        const int64_t x = (e.fm - rm) * 100;
        pm = x >= 0 ? div_floor_pos(x, e.am, e.inv_am) : x / e.am;
    }
    return (pc + pm) / 2;
}

constexpr uint32_t LA_MAX_WARPS = 8;     // 256-thread CTAs at most
constexpr uint32_t LA_FIRST_WINDOW = 8;  // tiles of the first window (then 32 per window)

template <int W>
__global__ void __launch_bounds__(256)
    k_least_alloc(const uint8_t* __restrict__ blobL, BitparLayout lay, const NodeEval* __restrict__ ev,
                  const float4* __restrict__ hint, const int64_t* __restrict__ ordL_s0, const int32_t* __restrict__ ordL_idx, PodView pv,
                  const uint2* __restrict__ rk, OutView ov, PeerOut po, const unsigned long long* __restrict__ live, uint32_t N) {
    const longlong2 amax = *reinterpret_cast<const longlong2*>(live + KS_MAX_LABEL_WORDS); // max allocatable cpu / memory
    __shared__ uint4 s_mask[LA_MAX_WARPS][32][2]; // per warp: the feasibility masks of the current window of tiles
    __shared__ int64_t s_top[LA_MAX_WARPS][32];   //           and the score bound of the first slot of each of them
    const uint32_t lane = threadIdx.x & 31, wq = lane & 7, quarter = lane >> 3, wid = threadIdx.x >> 5;
    const uint32_t warps = gridDim.x * (blockDim.x >> 5);
    uint32_t ne = 0;
    if (blockIdx.x == 0 && threadIdx.x == 0) exchange_stamp(po, 0);
    if (threadIdx.x == 0) trace_start(TR_ARGMAX1_START);
    for (uint32_t p = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); p < pv.P; p += warps) {
        const uint2 r = __ldg(rk + p);
        const PodThreshold t = pod_threshold(blobL, lay, r);
        unsigned long long sel[W];
        bool dead = r.x >= N || r.y >= N; // the request exceeds every node's free cpu / memory
#pragma unroll
        for (int w = 0; w < W; w++) {
            sel[w] = __ldg(pv.sel + (size_t)p * W + w);
            dead |= (sel[w] & ~__ldg(live + w)) != 0; // a required pair that no node carries
        }
        const int64_t rc = __ldg(pv.req_cpu + p), rm = __ldg(pv.req_mem + p);
        const float rcf = (float)rc, rmf = (float)rm;
        const bool rc_exact = rc > -(1ll << 24) && rc < (1ll << 24); // (float)rc is rc
        const bool bounded = rc >= 0 && rm >= 0; // else the bound does not hold: no early exit
        // per-pod slack: floor((f-r)*100/a) <= floor(f*100/a) - floor(r*100/a) and a <= a_max, so every feasible cell
        // scores <= bound(n) - D with D = (rc*100/ac_max + rm*100/am_max) / 2
        const int64_t D = bounded ? ((amax.x > 0 ? (rc * 100) / amax.x : 0) + (amax.y > 0 ? (rm * 100) / amax.y : 0)) / 2 : 0;
        int64_t best = INT64_MIN;
        int32_t bidx = -1;
        // The scan runs in windows of tiles: 8 tiles first (93 % of the pods of BASELINE C3 are done within them), then 32 at a
        // time.  Phase A: lane j derives the feasibility mask of tile k0 + j - the lanes work on DIFFERENT tiles, so the two
        // dependent rounds of table loads of a whole window overlap - and parks it in shared memory with the tile's top bound.
        // Phase B: the tiles that have a feasible slot at all are scored one by one, in bound order, by the whole warp.  Tiles
        // without a feasible slot cost nothing beyond phase A (a pod that fits nowhere no longer pays a full iteration per tile),
        // and the early exit is only evaluated in front of a tile that could change the result: the bounds descend, so it fires
        // there whenever it would have fired in front of an empty tile before it.
        uint32_t k0 = 0, win = LA_FIRST_WINDOW;
        bool done = dead;
        while (!done && k0 < lay.nt) {
            if (k0 > 0 && bounded && bidx >= 0 && best > __ldg(ordL_s0 + (size_t)k0 * BP_TILE) - D) break; // warp-uniform
            {
                uint32_t m[8] = {0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u};
                int64_t top = INT64_MIN;
                const uint32_t kt = k0 + lane;
                if (lane < win && kt < lay.nt) {
                    ptile_mask<W>(blobL, lay, t, sel, kt, m);
                    top = __ldg(ordL_s0 + (size_t)kt * BP_TILE);
                }
                s_mask[wid][lane][0] = make_uint4(m[0], m[1], m[2], m[3]);
                s_mask[wid][lane][1] = make_uint4(m[4], m[5], m[6], m[7]);
                s_top[wid][lane] = top;
                ne = __ballot_sync(0xffffffffu, (m[0] | m[1] | m[2] | m[3] | m[4] | m[5] | m[6] | m[7]) != 0u);
            }
            __syncwarp();
            while (ne) {
                const uint32_t j = __ffs(ne) - 1;
                ne &= ne - 1;
                const uint32_t k = k0 + j;
                if (bounded && bidx >= 0 && best > s_top[wid][j] - D) { // warp-uniform: nothing from here on can win or tie
                    done = true;
                    break;
                }
                // this lane's share of the tile's feasible slots: word wq, bit positions congruent to `quarter` mod 4
                const uint32_t bits = reinterpret_cast<const uint32_t*>(&s_mask[wid][j][0])[wq] & (0x11111111u << quarter);
                // Scores in single precision (k_build_eval): per feasible slot of this lane an interval [lo, hi] of integers that
                // contains the exact score - lo == hi (the score is KNOWN) unless the memory quotient lies within its error bound of
                // an integer, and [-inf, +inf] when the numbers leave the range in which the float arithmetic below is exact.  The
                // tile's winner scores >= max(lo), so only slots with hi >= max(max(lo), best so far) can win or tie: they load the
                // 4-byte node index (score known) or the 64-byte evaluation row for the exact 64-bit arithmetic (score not known).
                float hi[8];
                uint32_t known = 0; // bit i: lo == hi for this lane's i-th slot
                float lmax = -INFINITY;
#pragma unroll
                for (int i = 0; i < 8; i++) {
                    const uint32_t b = quarter + 4u * i;
                    const bool f = (bits >> b) & 1u;
                    const float4 h = f ? __ldg(hint + (size_t)k * BP_TILE + wq * 32 + b) : make_float4(0.f, 1.f, 0.f, 0.f);
                    const float x = (h.x - rcf) * 100.0f;           // exact while it is an integer below 2^24
                    const float pc = floorf(__fdiv_rn(x, h.y));     // = floor((free_cpu - rc) * 100 / alloc_cpu); 0 for y = +inf
                    const float tm = rmf * h.w, qm = h.z - tm;      // memory quotient, real-valued estimate
                    const float em = 2e-6f * (fabsf(h.z) + fabsf(tm)) + 1e-3f;
                    const float pm_lo = h.w == 0.f ? 0.f : floorf(qm - em), pm_hi = h.w == 0.f ? 0.f : floorf(qm + em);
                    // every float sum below must be exact: integers under 2^23
                    const bool ok = rc_exact && x >= 0.f && x < 16777216.f && pc < 4.0e6f && fabsf(qm) + em < 4.0e6f; // false for NaN
                    const float lo = floorf((pc + pm_lo) * 0.5f);
                    hi[i] = f ? (ok ? floorf((pc + pm_hi) * 0.5f) : INFINITY) : -INFINITY;
                    if (f && ok) {
                        lmax = fmaxf(lmax, lo);
                        known |= (lo == hi[i] ? 1u : 0u) << i;
                    }
                }
#pragma unroll
                for (int off = 16; off > 0; off >>= 1) lmax = fmaxf(lmax, __shfl_xor_sync(0xffffffffu, lmax, off));
                bool changed = false;
#pragma unroll
                for (int i = 0; i < 8; i++) {
                    const uint32_t b = quarter + 4u * i;
                    if (!((bits >> b) & 1u)) continue;              // not feasible
                    if (hi[i] < lmax) continue;                     // cannot reach the tile's winner
                    if (bidx >= 0 && hi[i] < (float)best) continue; // cannot reach the best so far (merged or this lane's)
                    const size_t slot = (size_t)k * BP_TILE + wq * 32 + b;
                    int64_t sc;
                    int32_t ni;
                    if ((known >> i) & 1u) {
                        sc = (int64_t)hi[i];
                        ni = __ldg(ordL_idx + slot);
                    } else {
                        const NodeEval e = ev[slot];
                        sc = least_alloc_score(e, rc, rm);
                        ni = e.idx;
                    }
                    if (sc > best || (sc == best && ni < bidx)) {
                        best = sc;
                        bidx = ni;
                        changed = true;
                    }
                }
                // every lane starts a tile with the same (best, bidx); merge only when some lane improved on it
                if (__any_sync(0xffffffffu, changed)) { // every lane ends with the tile-merged best
                    const Candidate w = warp_argmax(best, bidx);
                    best = w.key;
                    bidx = w.idx;
                }
            }
            __syncwarp(); // the next window overwrites this warp's slice of s_mask / s_top
            k0 += win;
            win = 32;
        }
        if (lane == 0) store_binding(ov, po, p, bidx, bidx >= 0 ? best : 0);
    }
    if (c_trace) {
        __syncthreads();
        if (threadIdx.x == 0) trace_end(TR_ARGMAX1_END);
    }
    exchange_signal(po);
}

// ------------------------------------------------------------------------------------------------ host side
static uint32_t round16(uint32_t x) { return (x + 15u) & ~15u; }

static uint64_t per_tile_bytes(uint32_t nb, uint32_t W) {
    return (uint64_t)nb * 20 + 2ull * BP_TABLE_BYTES + 64ull * W * 32 + 64ull * W * 16; // last term: pair-column skew
    // (tables are allocated per quad of tiles: make_layout_smem re-checks the exact blob size)
}

static bool fill_offsets(BitparLayout* lay, uint32_t W) {
    const uint64_t nb = lay->nb, nt = lay->nt;
    if (per_tile_bytes(lay->nb, W) * nt + 1024 > 0xF0000000ull) return false;
    uint32_t off = 0;
    lay->off_baseC = off;
    off += round16((uint32_t)(nb * nt * 2));
    lay->off_baseM = off;
    off += round16((uint32_t)(nb * nt * 2));
    lay->off_membC = off;
    off += round16((uint32_t)(nb * nt * 8));
    lay->off_membM = off;
    off += round16((uint32_t)(nb * nt * 8));
    off = (off + 127u) & ~127u; // table lines are 128 bytes
    lay->off_tabC = off;
    off += table_area_bytes((uint32_t)nt);
    lay->off_tabM = off;
    off += table_area_bytes((uint32_t)nt);
    lay->off_pairs = off;
    lay->pstride = pair_stride((uint32_t)nt);
    off += 64u * W * lay->pstride;
    lay->blob_bytes = (off + 127u) & ~127u;
    return true;
}

// "rows" format (ks_bitpar.h): column blocks of RW_TILES tiles; the pair columns are staged with the tables when
// everything fits in shared memory (W <= 4), else they are read through L1/L2
static bool make_layout_rows(uint32_t N, uint32_t W, RowsLayout* lay) {
    const uint32_t n_tiles = (N + BP_TILE - 1) / BP_TILE;
    if (n_tiles == 0) return false;
    lay->n_tiles = n_tiles;
    lay->ncb = (n_tiles + RW_TILES - 1) / RW_TILES;
    lay->off_tabC = 0;
    lay->off_tabM = RW_TAB_BYTES;
    lay->off_pairs = 2 * RW_TAB_BYTES;
    const uint32_t pairs_bytes = 64u * W * RW_LINE;
    lay->cb_stride = 2 * RW_TAB_BYTES + pairs_bytes; // multiple of 256
    lay->pairs_smem = lay->cb_stride <= (uint32_t)BP_SMEM_MAX - 1024u ? 1u : 0u;
    lay->smem_bytes = lay->pairs_smem ? lay->cb_stride : 2 * RW_TAB_BYTES;
    lay->n_thr = N + 1;
    // rank tables: 2 x ncb x (N+1) x 16 B; beyond 4 GB the per-cell kernel serves the snapshot
    return (uint64_t)lay->ncb * lay->n_thr * RW_TILES * 2ull * 2ull <= (4ull << 30);
}

// flat layout for the priority-ordered index (global memory, all tiles in one blob)
static bool make_layout_flat(uint32_t N, uint32_t W, BitparLayout* lay) {
    lay->nb = (N >> 6) + 1;
    lay->ncb = 1;
    lay->nt = (N + BP_TILE - 1) / BP_TILE;
    return lay->nt > 0 && fill_offsets(lay, W);
}

static std::atomic<uint64_t> g_regrow_epoch{0}; // any reallocation invalidates cached CUDA graphs (BitparIndex::epoch)
template <class T>
static cudaError_t regrow(T*& p, size_t count) {
    if (p) cudaFree(p);
    p = nullptr;
    g_regrow_epoch++;
    return cudaMalloc(reinterpret_cast<void**>(&p), count * sizeof(T));
}

void bitpar_release(BitparIndex& ix) {
    void* ptrs[] = {ix.sortedC, ix.sortedM, ix.gposC, ix.gposM, ix.ord_prio,
                    ix.ord_idx, ix.splC,  ix.splM,  ix.blobP,    ix.pod_ranks, ix.tail_list,
                    ix.rk_hist, ix.rk_spl_v, ix.rk_spl_i, ix.rk_bkt, ix.rk_loc, ix.rk_perm, ix.rec_s,
                    ix.blobR,   ix.rank,   ix.tile_sorted, ix.ordL_s0, ix.ordL_idx, ix.evalL, ix.hintL, ix.blobL, ix.live, ix.cursor};
    for (void* p : ptrs)
        if (p) cudaFree(p);
    if (ix.trace) {
        unsigned long long* none = nullptr;
        cudaMemcpyToSymbol(c_trace, &none, sizeof(none));
        cudaFree(ix.trace);
    }
    if (ix.aux) cudaStreamDestroy(ix.aux);
    if (ix.ev_fork) cudaEventDestroy(ix.ev_fork);
    if (ix.ev_join) cudaEventDestroy(ix.ev_join);
    ix = BitparIndex();
}

cudaError_t bitpar_build(BitparIndex& ix, const NodeTable& nt, int64_t* prio, cudaStream_t st) {
    ix.valid = false;
    ix.N = nt.N;
    ix.W = nt.W;
    if (nt.N == 0) return cudaSuccess;
    const uint32_t Nord = ((nt.N + BP_TILE - 1) / BP_TILE) * BP_TILE;
    ix.Nord = Nord;
    cudaError_t e;
    if (Nord > ix.cap_nodes) {
        const size_t cap = Nord + Nord / 8 + BP_TILE;
        if ((e = regrow(ix.sortedC, cap)) != cudaSuccess) return e;
        if ((e = regrow(ix.sortedM, cap)) != cudaSuccess) return e;
        if ((e = regrow(ix.gposC, cap)) != cudaSuccess) return e;
        if ((e = regrow(ix.gposM, cap)) != cudaSuccess) return e;
        if ((e = regrow(ix.ord_prio, cap)) != cudaSuccess) return e;
        if ((e = regrow(ix.ord_idx, cap)) != cudaSuccess) return e;
        if ((e = regrow(ix.splC, RANK_SPLITTERS)) != cudaSuccess) return e;
        if ((e = regrow(ix.splM, RANK_SPLITTERS)) != cudaSuccess) return e;
        if ((e = regrow(ix.rk_bkt, N_ORDERS * cap)) != cudaSuccess) return e;
        if ((e = regrow(ix.rk_loc, N_ORDERS * cap)) != cudaSuccess) return e;
        if ((e = regrow(ix.rk_perm, N_ORDERS * cap)) != cudaSuccess) return e;
        if ((e = regrow(ix.ordL_s0, cap)) != cudaSuccess) return e;
        if ((e = regrow(ix.ordL_idx, cap)) != cudaSuccess) return e;
        if ((e = regrow(ix.evalL, cap)) != cudaSuccess) return e;
        if ((e = regrow(ix.hintL, cap)) != cudaSuccess) return e;
        ix.cap_nodes = cap;
    }
    uint32_t stride = 1;
    while ((nt.N + stride - 1) / stride > (uint32_t)RANK_SPLITTERS) stride <<= 1;
    ix.spl_stride = stride;
    ix.n_spl = (nt.N + stride - 1) / stride;
    if (!ix.rk_hist) {
        if ((e = regrow(ix.rk_hist, N_ORDERS * RANK_BUCKETS)) != cudaSuccess) return e;
        if ((e = regrow(ix.rk_spl_v, N_ORDERS * RANK_BUCKETS)) != cudaSuccess) return e;
        if ((e = regrow(ix.rk_spl_i, N_ORDERS * RANK_BUCKETS)) != cudaSuccess) return e;
    }
    if (!ix.live) {
        if ((e = regrow(ix.live, KS_MAX_LABEL_WORDS + 2)) != cudaSuccess) return e; // + max allocatable cpu, memory
    }
    if ((e = cudaMemsetAsync(ix.live, 0, (KS_MAX_LABEL_WORDS + 2) * 8, st)) != cudaSuccess) return e;
    k_node_bound<<<(nt.N + 255) / 256, 256, 0, st>>>(nt, prio + nt.Npad, ix.live);
    g_launches++;
    k_node_splitters<<<N_ORDERS, RANK_SAMPLES, 0, st>>>(nt, prio, ix.rk_spl_v, ix.rk_spl_i, ix.rk_hist);
    k_node_bucket<<<(nt.N + 255) / 256, 256, 0, st>>>(nt, prio, ix.rk_spl_v, ix.rk_spl_i, ix.rk_hist, ix.rk_bkt, ix.rk_loc);
    k_node_scatter<<<(nt.N + 255) / 256, 256, 0, st>>>(nt.N, ix.rk_hist, ix.rk_bkt, ix.rk_loc, ix.rk_perm);
    k_node_rank<<<(Nord + 255) / 256, 256, 0, st>>>(nt, prio, ix.rk_hist, ix.rk_bkt, ix.rk_perm, ix.sortedC, ix.sortedM,
                                                    ix.gposC, ix.gposM, ix.ord_prio, ix.ord_idx, Nord, ix.splC, ix.splM,
                                                    stride, ix.ordL_s0, ix.ordL_idx);
    g_launches += 4;
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    BitparLayout layP{};
    if (!make_layout_flat(nt.N, nt.W, &layP)) return cudaSuccess; // direct path only
    if (layP.blob_bytes > ix.cap_blobP) {
        const size_t cap = (size_t)layP.blob_bytes + layP.blob_bytes / 8;
        if ((e = regrow(ix.blobP, cap)) != cudaSuccess) return e;
        if ((e = regrow(ix.blobL, cap)) != cudaSuccess) return e;
        ix.cap_blobP = cap;
    }
    {
        RowsLayout lr{};
        if (!make_layout_rows(nt.N, nt.W, &lr)) return cudaSuccess; // direct path only
        const size_t need = (size_t)lr.ncb * lr.cb_stride;
        if (need > ix.cap_blobR) {
            if ((e = regrow(ix.blobR, need + need / 8)) != cudaSuccess) return e;
            ix.cap_blobR = need + need / 8;
        }
        const size_t need_rank = (size_t)lr.ncb * lr.n_thr * 2 * RW_TILES;
        if (need_rank > ix.cap_rank) {
            const size_t cap = need_rank + need_rank / 8;
            if ((e = regrow(ix.rank, cap)) != cudaSuccess) return e;
            ix.cap_rank = cap;
        }
        if (lr.ncb > ix.cap_cursor) { // one work cursor per column block (k_mask_rows)
            if ((e = regrow(ix.cursor, ((size_t)lr.ncb + 64) * RW_CURSOR_STRIDE)) != cudaSuccess) return e;
            ix.cap_cursor = (size_t)lr.ncb + 64;
        }
        const size_t need_ts = 2ull * lr.ncb * RW_TILES * BP_TILE;
        if (need_ts > ix.cap_tsorted) {
            if ((e = regrow(ix.tile_sorted, need_ts + need_ts / 8)) != cudaSuccess) return e;
            ix.cap_tsorted = need_ts + need_ts / 8;
        }
        k_build_cbtile<<<lr.ncb * RW_TILES, 288, 0, st>>>(nt, ix.gposC, ix.gposM, ix.blobR, lr, ix.tile_sorted);
        g_launches++;
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
        k_build_ranks<<<dim3((lr.n_thr + 255) / 256, lr.ncb), 256, 0, st>>>(ix.tile_sorted, lr, ix.rank);
        g_launches++;
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
        ix.lay_r = lr;
    }
    k_build_tile<<<layP.nt, 288, 0, st>>>(nt, ix.gposC, ix.gposM, ix.ord_idx, ix.blobP, layP);
    g_launches++;
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    // KS_SCORE_LEAST_ALLOCATED: the same flat index in descending order of the score bound + per-slot evaluation rows
    k_build_tile<<<layP.nt, 288, 0, st>>>(nt, ix.gposC, ix.gposM, ix.ordL_idx, ix.blobL, layP);
    k_build_eval<<<(Nord + 255) / 256, 256, 0, st>>>(nt, ix.ordL_idx, Nord, ix.evalL, ix.hintL);
    g_launches += 2;
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    ix.layP = layP;
    ix.valid = true;
    ix.epoch = g_regrow_epoch.load();
    return cudaSuccess;
}

bool bitpar_profitable(const BitparIndex& ix, uint32_t P) {
    // below ~16M cells the per-call rank pass and blob staging outweigh the per-cell kernel;
    // the mask kernel indexes (pod, tile) items with 32 bits
    return ix.valid && (uint64_t)P * ix.N >= (1ull << 24) && (uint64_t)P * RW_TILES < (1ull << 31);
}

template <int W, int THREADS>
static cudaError_t set_smem_attr1() {
    return cudaFuncSetAttribute(k_mask_rows<W, W <= 4, THREADS>, cudaFuncAttributeMaxDynamicSharedMemorySize, BP_SMEM_MAX - 1024);
}
template <int W>
static cudaError_t set_smem_attr() {
    cudaError_t e;
    if ((e = set_smem_attr1<W, 896>()) != cudaSuccess) return e;
    return set_smem_attr1<W, 960>();
}

// everything that allocates or configures: must run before a (possibly stream-captured) bitpar_select
cudaError_t bitpar_prepare(BitparIndex& ix, uint32_t P) {
    cudaError_t e;
    if (!ix.valid) return cudaErrorNotSupported;
    if (ix.sms == 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&ix.sms, cudaDevAttrMultiProcessorCount, dev);
        if ((e = cudaStreamCreateWithFlags(&ix.aux, cudaStreamNonBlocking)) != cudaSuccess) return e;
        if ((e = cudaEventCreateWithFlags(&ix.ev_fork, cudaEventDisableTiming)) != cudaSuccess) return e;
        if ((e = cudaEventCreateWithFlags(&ix.ev_join, cudaEventDisableTiming)) != cudaSuccess) return e;
        if ((e = set_smem_attr<1>()) != cudaSuccess) return e;
        if ((e = set_smem_attr<2>()) != cudaSuccess) return e;
        if ((e = set_smem_attr<4>()) != cudaSuccess) return e;
        if ((e = set_smem_attr<8>()) != cudaSuccess) return e;
        if ((e = cudaFuncSetAttribute(k_pod_ranks, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      RANK_SPLITTERS * 2 * (int)sizeof(int64_t))) != cudaSuccess)
            return e;
        const char* tr = getenv("KS_TRACE");
        if (tr && tr[0] == '1') { // one trace buffer per device: the most recently prepared index owns the stamps
            if ((e = cudaMalloc(&ix.trace, BP_TRACE_WORDS * sizeof(unsigned long long))) != cudaSuccess) return e;
            if ((e = cudaMemset(ix.trace, 0, BP_TRACE_WORDS * sizeof(unsigned long long))) != cudaSuccess) return e;
            if ((e = cudaMemcpyToSymbol(c_trace, &ix.trace, sizeof(ix.trace))) != cudaSuccess) return e;
        }
    }
    if (P > ix.cap_pods) {
        const size_t cap = (size_t)P + P / 8 + 64;
        if ((e = regrow(ix.pod_ranks, cap)) != cudaSuccess) return e;
        if ((e = regrow(ix.tail_list, cap + 1)) != cudaSuccess) return e; // [cap] = the list length counter
        if ((e = regrow(ix.rec_s, cap + 8)) != cudaSuccess) return e;
        ix.cap_pods = cap;
    }
    ix.epoch = g_regrow_epoch.load();
    return cudaSuccess;
}

template <int W>
static cudaError_t select_w(BitparIndex& ix, SelectLaunch& L, cudaEvent_t before_mask, cudaEvent_t after_mask) {
    cudaError_t e;
    const uint32_t P = L.pv.P;
    if ((uint64_t)P * RW_TILES >= (1ull << 31)) return cudaErrorInvalidValue;
    if ((e = bitpar_prepare(ix, P)) != cudaSuccess) return e; // no-op when the caller prepared already
    const bool need_mask_pass = L.ov.mask || L.ov.cnt;
    const int sms = ix.sms;
    if (ix.trace)
        if ((e = cudaMemsetAsync(ix.trace, 0, BP_TRACE_WORDS * sizeof(unsigned long long), L.stream)) != cudaSuccess) return e;
    // one 1024-thread CTA per SM (splitters in dynamic shared memory); two pods per thread and pass once P > #SMs * 1024
    const uint32_t rank_grid = (uint32_t)std::min<uint64_t>((uint64_t)sms, ((uint64_t)P + RANK_THREADS - 1) / RANK_THREADS);
    const size_t rank_smem = (size_t)ix.n_spl * 2 * sizeof(int64_t);
    const bool want_bind = L.ov.node_idx || L.ov.score;
    const bool overlap_bind = before_mask == nullptr && after_mask == nullptr;
    // How the mask kernel (persistent, one CTA per SM, SM-bound: every SM it does not get costs it 1/#SMs) and the argmax
    // kernels (latency-bound, ~15 us + 45 ns per 1000 pods on their own) share the chip.  Inside a CUDA graph the mask
    // kernel gets the SMs first, and a 256-thread argmax CTA does not fit beside a mask CTA (registers), so by default the
    // argmax kernels run after it (profiles/r02_experiments.txt, sessions G-I).
    //   * short mask pass (< 256 MB of mask, ~60 us): the mask kernel leaves one SM in six to the argmax kernels, which then
    //     run beside it from the start; what they (and the exchange behind them) would add at the end costs more than the SMs.
    //   * long mask pass with an exchange attached: 896-thread mask CTAs + 128-thread argmax CTAs, which do fit beside them:
    //     the bindings go out to the peers early and the ~18 us of fences / flag latency hide under the mask kernel (the mask
    //     kernel pays for the company roughly what the argmax kernels cost alone, so without an exchange this buys nothing).
    //   * long mask pass, no exchange: 960-thread mask CTAs (fastest), argmax kernels behind them.
    const uint64_t mask_bytes = (uint64_t)P * (L.ov.mask ? L.ov.mask_row_words * 4ull : (uint64_t)ix.lay_r.n_tiles * 32ull);
    // (timing mode keeps the same shapes; it only moves the argmax kernels behind the mask kernel)
    const bool short_pass = need_mask_pass && want_bind && mask_bytes < (256ull << 20) && sms >= 48;
    const bool beside = !short_pass && need_mask_pass && want_bind && L.po.n > 0;
    const int threads = beside ? 896 : 960;
    const uint32_t at = beside ? 128u : 256u; // threads per argmax CTA
    const uint32_t mask_sms = short_pass ? (uint32_t)(sms - sms / 6) : (uint32_t)sms;
    const uint32_t n_groups = (P + 7) / 8;
    const uint64_t F = (uint64_t)n_groups * ix.lay_r.ncb;
    const uint32_t warps = (uint32_t)threads / 32;
    const uint32_t mask_grid = (uint32_t)std::min<uint64_t>((uint64_t)mask_sms, (F + warps - 1) / warps);
    k_pod_ranks<<<rank_grid, RANK_THREADS, rank_smem, L.stream>>>(L.pv, ix.sortedC, ix.sortedM, ix.N, ix.splC, ix.splM, ix.n_spl, ix.spl_stride,
                                                 ix.pod_ranks, (need_mask_pass && ix.lay_r.ncb > 1) ? L.ov.cnt : nullptr, ix.W,
                                                 need_mask_pass ? ix.rec_s : nullptr, ix.cursor, need_mask_pass ? ix.lay_r.ncb : 0u);
    g_launches++;
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    // argmax scan (needs only the pod ranks) on an auxiliary stream, forked here.  In timing mode it is enqueued on the main
    // stream behind the mask kernel instead, so that the event pair around the mask kernel times that kernel alone.
    if (want_bind) {
        if ((e = cudaEventRecord(ix.ev_fork, L.stream)) != cudaSuccess) return e;
        if ((e = cudaStreamWaitEvent(ix.aux, ix.ev_fork, 0)) != cudaSuccess) return e;
    }
    auto enqueue_bind = [&](cudaStream_t bs) -> cudaError_t {
        uint32_t* tail_count = ix.tail_list + ix.cap_pods;
        if ((e = cudaMemsetAsync(tail_count, 0, sizeof(uint32_t), bs)) != cudaSuccess) return e;
        if (L.policy == KS_SCORE_LEAST_ALLOCATED) {
            const uint32_t wpc = at / 32; // one warp per pod
            const uint32_t grid = (uint32_t)std::min<uint64_t>((uint64_t)sms * (2048 / at), ((uint64_t)P + wpc - 1) / wpc);
            k_least_alloc<W><<<grid, at, 0, bs>>>(ix.blobL, ix.layP, ix.evalL, ix.hintL, ix.ordL_s0, ix.ordL_idx, L.pv, ix.pod_ranks, L.ov, L.po, ix.live,
                                                  ix.N);
            g_launches++;
            if ((e = cudaGetLastError()) != cudaSuccess) return e;
        } else {
            const bool has_tail = ix.layP.nt > FF_HEAD_TILES;
            k_first_fit_head<W><<<(P + at - 1) / at, at, 0, bs>>>(ix.blobP, ix.layP, ix.ord_idx, ix.ord_prio, L.pv, ix.pod_ranks, L.ov,
                                                                 ix.tail_list, tail_count, L.po, !has_tail, ix.live, ix.N);
            g_launches++;
            if ((e = cudaGetLastError()) != cudaSuccess) return e;
            if (has_tail) {
                k_first_fit_tail<W><<<sms * (512 / at), at, 0, bs>>>(ix.blobP, ix.layP, ix.ord_idx, ix.ord_prio, L.pv, ix.pod_ranks, L.ov,
                                                             ix.tail_list, tail_count, L.po);
                g_launches++;
                if ((e = cudaGetLastError()) != cudaSuccess) return e;
            }
        }
        // bindings are final here: start their device-to-host copy now, under the mask kernel
        if (L.host_node_idx && L.ov.node_idx) {
            if ((e = cudaMemcpyAsync(L.host_node_idx, L.ov.node_idx, (size_t)P * 4, cudaMemcpyDeviceToHost, bs)) != cudaSuccess) return e;
            L.host_node_idx = nullptr;
        }
        if (L.host_score && L.ov.score) {
            if ((e = cudaMemcpyAsync(L.host_score, L.ov.score, (size_t)P * 8, cudaMemcpyDeviceToHost, bs)) != cudaSuccess) return e;
            L.host_score = nullptr;
        }
        if (L.ready_event) { // tell the caller that node_idx / score are final (the mask pass may still be running)
            if ((e = record_ready_event(L.ready_event, bs)) != cudaSuccess) return e;
            L.ready_event = nullptr;
        }
        return cudaSuccess;
    };
    if (want_bind && overlap_bind)
        if ((e = enqueue_bind(ix.aux)) != cudaSuccess) return e;
    if (need_mask_pass) {
        if (before_mask)
            if ((e = cudaEventRecord(before_mask, L.stream)) != cudaSuccess) return e;
        RowsParams prm;
        prm.blob = ix.blobR;
        prm.lay = ix.lay_r;
        prm.rank = ix.rank;
        prm.rec_s = ix.rec_s;
        prm.sel_s = reinterpret_cast<const unsigned long long*>(L.pv.sel); // pod order: the caller's selector words
        prm.n_groups = n_groups;
        prm.mask = L.ov.mask;
        prm.row_words = (uint32_t)L.ov.mask_row_words;
        prm.cnt = L.ov.cnt;
        prm.cursor = ix.cursor;
        void (*kern)(RowsParams) = threads == 896 ? k_mask_rows<W, W <= 4, 896> : k_mask_rows<W, W <= 4, 960>;
        kern<<<mask_grid, threads, ix.lay_r.smem_bytes, L.stream>>>(prm);
        g_launches++;
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
        if (after_mask)
            if ((e = cudaEventRecord(after_mask, L.stream)) != cudaSuccess) return e;
    } else if (before_mask) {
        if ((e = cudaEventRecord(before_mask, L.stream)) != cudaSuccess) return e;
    }
    if (want_bind && !overlap_bind) // timing mode: on the main stream, behind the mask kernel
        if ((e = enqueue_bind(L.stream)) != cudaSuccess) return e;
    if (want_bind) { // join the auxiliary stream (it holds the argmax kernels unless timing mode put them on the main one)
        if ((e = cudaEventRecord(ix.ev_join, ix.aux)) != cudaSuccess) return e;
        if ((e = cudaStreamWaitEvent(L.stream, ix.ev_join, 0)) != cudaSuccess) return e;
    }
    if (after_mask && !need_mask_pass)
        if ((e = cudaEventRecord(after_mask, L.stream)) != cudaSuccess) return e;
    return cudaSuccess;
}

cudaError_t bitpar_read_trace(const BitparIndex& ix, unsigned long long out_ns[BP_TRACE_WORDS]) {
    if (!ix.trace) return cudaErrorNotSupported;
    cudaError_t e = cudaDeviceSynchronize();
    if (e != cudaSuccess) return e;
    if ((e = cudaMemcpy(out_ns, ix.trace, BP_TRACE_WORDS * sizeof(unsigned long long), cudaMemcpyDeviceToHost)) != cudaSuccess) return e;
    if (out_ns[TR_MASK_FIRST_CTA_END_INV]) out_ns[TR_MASK_FIRST_CTA_END_INV] = ~out_ns[TR_MASK_FIRST_CTA_END_INV];
    return cudaSuccess;
}

cudaError_t bitpar_select(BitparIndex& ix, SelectLaunch& L, cudaEvent_t before_mask, cudaEvent_t after_mask) {
    if (!ix.valid) return cudaErrorNotSupported;
    switch (ix.W) {
        case 1: return select_w<1>(ix, L, before_mask, after_mask);
        case 2: return select_w<2>(ix, L, before_mask, after_mask);
        case 4: return select_w<4>(ix, L, before_mask, after_mask);
        case 8: return select_w<8>(ix, L, before_mask, after_mask);
        default: return cudaErrorInvalidValue;
    }
}

} // namespace ks
