// ks_direct.cu — per-cell ("direct") kernels for sm_100a.
//   K0  k_node_free_reduce     free = alloc - sum(bound)            /root/reference/src/predicates.rs:27-38
//   K1  k_check_cells          2-bit reason code per cell           /root/reference/src/predicates.rs:63-77
//   K2d k_select_direct        fused feasible mask + count + argmax score, node tiles staged through
//                              shared memory by TMA bulk copies (cp.async.bulk + mbarrier), one lane per
//                              node, warp ballot packs 32 cells into one mask word, warp-shuffle argmax.
// The per-cell kernel is the generic path (any score policy, any P); ks_bitpar.cu holds the bit-parallel
// fast path that the headline configuration uses.
#include "ks_internal.cuh"
#include "ks_launch.h"

#include <algorithm>

namespace ks {

std::atomic<uint64_t> g_launches{0};

// ------------------------------------------------------------------------------------------------ K0
__global__ void k_node_free_reduce(int64_t* __restrict__ free_cpu, int64_t* __restrict__ free_mem,
                                   const int32_t* __restrict__ bnode, const int64_t* __restrict__ bcpu,
                                   const int64_t* __restrict__ bmem, uint64_t B) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (; i < B; i += stride) {
        int32_t n = bnode[i];
        // integer adds commute -> result is deterministic regardless of atomic order (util.rs:31-36)
        atomicAdd(reinterpret_cast<unsigned long long*>(free_cpu + n), (unsigned long long)(-bcpu[i]));
        atomicAdd(reinterpret_cast<unsigned long long*>(free_mem + n), (unsigned long long)(-bmem[i]));
    }
}

cudaError_t launch_free_reduce(int64_t* free_cpu, int64_t* free_mem, const int32_t* bnode, const int64_t* bcpu,
                               const int64_t* bmem, uint64_t B, cudaStream_t st) {
    if (B == 0) return cudaSuccess;
    int threads = 256;
    uint64_t blocks = (B + threads - 1) / threads;
    if (blocks > 4096) blocks = 4096; // grid-stride beyond that
    k_node_free_reduce<<<(unsigned)blocks, threads, 0, st>>>(free_cpu, free_mem, bnode, bcpu, bmem, B);
    g_launches++;
    return cudaGetLastError();
}

// range check of free values + static node priority for KS_SCORE_LEFTOVER (leftover_prio)
__global__ void k_node_prio(const int64_t* __restrict__ free_cpu, const int64_t* __restrict__ free_mem,
                            int64_t* __restrict__ prio, uint32_t N, uint32_t Npad, int* __restrict__ range_flag) {
    uint32_t n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= Npad) return;
    if (n >= N) {
        prio[n] = INT64_MIN;
        return;
    }
    int64_t fc = free_cpu[n], fm = free_mem[n];
    const int64_t LC = KS_MAX_CPU_MILLI, LM = KS_MAX_MEM_BYTES; // keeps prio and (free-req)*100 inside int64
    if (fc > LC || fc < -LC || fm > LM || fm < -LM) {
        atomicExch(range_flag, 1);
        prio[n] = INT64_MIN + 1;
        return;
    }
    prio[n] = leftover_prio(fc, fm);
}

cudaError_t launch_node_prio(const int64_t* free_cpu, const int64_t* free_mem, int64_t* prio, uint32_t N,
                             uint32_t Npad, int* range_flag, cudaStream_t st) {
    k_node_prio<<<(Npad + 255) / 256, 256, 0, st>>>(free_cpu, free_mem, prio, N, Npad, range_flag);
    g_launches++;
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------ exchange
// ks_exchange (include/ksched.h).  The bit-parallel path stores the bindings into the peers' gather buffers from
// inside its argmax kernels (ks_bitpar.cu); the per-cell path pushes its finished arrays with this kernel.
__global__ void __launch_bounds__(256)
    k_exchange_push(PeerOut po, const int32_t* __restrict__ node_idx, const int64_t* __restrict__ score, uint32_t P) {
    if (blockIdx.x == 0 && threadIdx.x == 0) exchange_stamp(po, 0);
    for (uint32_t p = blockIdx.x * blockDim.x + threadIdx.x; p < P; p += gridDim.x * blockDim.x)
        store_binding(OutView{}, po, p, node_idx[p], score[p]);
    exchange_signal(po);
}

// One warp; lane r waits until rank r's flag carries this rank's current sequence number (all ranks step in
// lockstep).  A peer that never arrives raises *error_flag after ~4 s instead of hanging the GPU.
__global__ void __launch_bounds__(32) k_exchange_wait(PeerOut po, int* __restrict__ error_flag) {
    const uint32_t r = threadIdx.x;
    if (r == 0) exchange_stamp(po, 2);
    if (r < po.world && r != po.rank) {
        const uint32_t target = *reinterpret_cast<volatile uint32_t*>(po.state);
        unsigned long long t0;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
        for (;;) {
            uint32_t v;
            asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(po.local_flags + r) : "memory");
            if ((int32_t)(v - target) >= 0) break;
            unsigned long long t1;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
            if (t1 - t0 > 4000000000ull) {
                if (error_flag) atomicExch(error_flag, 2);
                break;
            }
            __nanosleep(200);
        }
    }
    __syncwarp();
    if (r == 0) exchange_stamp(po, 3);
}

cudaError_t launch_exchange_push(const PeerOut& po, const int32_t* node_idx, const int64_t* score, uint32_t P, cudaStream_t st) {
    if (po.n == 0) return cudaSuccess;
    const uint32_t grid = std::max(1u, std::min<uint32_t>(256u, (P + 255u) / 256u));
    k_exchange_push<<<grid, 256, 0, st>>>(po, node_idx, score, P);
    g_launches++;
    return cudaGetLastError();
}

cudaError_t launch_exchange_wait(const PeerOut& po, int* error_flag, cudaStream_t st) {
    if (po.n == 0) return cudaSuccess;
    k_exchange_wait<<<1, 32, 0, st>>>(po, error_flag);
    g_launches++;
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------ store ceiling
// What a kernel that ONLY writes can reach on this device (ks_measure_write_bandwidth): coalesced 256-bit stores,
// grid-stride, nothing else.  The mask kernel is compared with this next to the copy-based HBM peak (DESIGN.md section 7).
__global__ void __launch_bounds__(256) k_fill256(uint8_t* __restrict__ dst, uint64_t n32, uint32_t v) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n32; i += (uint64_t)gridDim.x * blockDim.x)
        asm volatile("st.global.v8.b32 [%0], {%1,%1,%1,%1,%1,%1,%1,%1};" ::"l"(dst + i * 32), "r"(v) : "memory");
}

cudaError_t launch_fill256(void* dst, uint64_t bytes, uint32_t v, int sms, cudaStream_t st) {
    k_fill256<<<sms * 8, 256, 0, st>>>(static_cast<uint8_t*>(dst), bytes / 32, v);
    g_launches++;
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------ K1
__device__ __forceinline__ int cell_code(int64_t rc, int64_t rm, const uint64_t* __restrict__ sel, int64_t fc,
                                         int64_t fm, const uint64_t* __restrict__ labels, uint32_t n,
                                         uint32_t Npad, uint32_t W) {
    bool fit = (rc <= fc) && (rm <= fm); // predicates.rs:42
    uint64_t miss = 0;
    for (uint32_t w = 0; w < W; w++) miss |= sel[w] & ~labels[(uint64_t)w * Npad + n];
    return !fit ? KS_CELL_NOT_ENOUGH_RESOURCES : (miss ? KS_CELL_NODE_SELECTOR_MISMATCH : KS_CELL_OK); // :68-76
}

__global__ void k_check_cells(NodeTable nt, PodView pv, uint8_t* __restrict__ codes, uint32_t node_begin,
                              uint32_t node_count) {
    uint64_t cell = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    uint64_t total = (uint64_t)pv.P * node_count;
    if (cell >= total) return;
    uint32_t p = (uint32_t)(cell / node_count);
    uint32_t n = node_begin + (uint32_t)(cell % node_count);
    codes[cell] = (uint8_t)cell_code(pv.req_cpu[p], pv.req_mem[p], pv.sel + (uint64_t)p * nt.W, nt.free_cpu[n],
                                     nt.free_mem[n], nt.labels, n, nt.Npad, nt.W);
}

cudaError_t launch_check_cells(const NodeTable& nt, const PodView& pv, uint8_t* codes, uint32_t node_begin,
                               uint32_t node_count, cudaStream_t st) {
    uint64_t total = (uint64_t)pv.P * node_count;
    if (total == 0) return cudaSuccess;
    uint64_t blocks = (total + 255) / 256;
    if (blocks > 0x7fffffffull) return cudaErrorInvalidValue;
    k_check_cells<<<(unsigned)blocks, 256, 0, st>>>(nt, pv, codes, node_begin, node_count);
    g_launches++;
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------ K1s
// The reference's own selection policy (/root/reference/src/main.rs:49-71) with a seeded generator: up to
// `attempts` uniform draws with replacement per pod, the first draw whose cell passes check_node_validity wins.
// One thread per pod; the node rows it touches are random gathers served by L2 (the node table is a few MB).
__device__ __forceinline__ uint64_t splitmix64_next(uint64_t& s) {
    uint64_t z = (s += 0x9E3779B97F4A7C15ull);
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}

__global__ void k_select_sampling(NodeTable nt, PodView pv, uint32_t attempts, uint64_t seed, uint64_t pod_offset,
                                  int32_t* __restrict__ node_idx, uint32_t* __restrict__ n_attempts,
                                  int32_t* __restrict__ draw_node, uint8_t* __restrict__ draw_code) {
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= pv.P) return;
    uint64_t state = KS_SAMPLING_STREAM(seed, pod_offset + p);
    const int64_t rc = pv.req_cpu[p], rm = pv.req_mem[p];
    const uint64_t* sel = pv.sel + (uint64_t)p * nt.W;
    int32_t chosen = -1;
    uint32_t a = 0;
    for (; a < attempts; a++) {                                         // main.rs:53
        const uint32_t n = (uint32_t)(splitmix64_next(state) % nt.N); // :56-57 choose()
        const int code = cell_code(rc, rm, sel, nt.free_cpu[n], nt.free_mem[n], nt.labels, n, nt.Npad, nt.W); // :61
        if (draw_node) draw_node[(uint64_t)p * attempts + a] = (int32_t)n;
        if (draw_code) draw_code[(uint64_t)p * attempts + a] = (uint8_t)code; // the reason main.rs:62 logs
        if (code == KS_CELL_OK) {                                     // :63-65
            chosen = (int32_t)n;
            a++;
            break;
        }
    }
    for (uint32_t r = a; r < attempts; r++) { // attempts never made
        if (draw_node) draw_node[(uint64_t)p * attempts + r] = -1;
        if (draw_code) draw_code[(uint64_t)p * attempts + r] = 0xff;
    }
    node_idx[p] = chosen;
    if (n_attempts) n_attempts[p] = a;
}

cudaError_t launch_select_sampling(const NodeTable& nt, const PodView& pv, uint32_t attempts, uint64_t seed,
                                   uint64_t pod_offset, int32_t* node_idx, uint32_t* n_attempts, int32_t* draw_node,
                                   uint8_t* draw_code, cudaStream_t st) {
    if (pv.P == 0) return cudaSuccess;
    k_select_sampling<<<(pv.P + 255) / 256, 256, 0, st>>>(nt, pv, attempts, seed, pod_offset, node_idx, n_attempts,
                                                          draw_node, draw_code);
    g_launches++;
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------ K2 direct
template <int W>
struct PodsPerWarp {
    static constexpr int v = W <= 2 ? 8 : (W == 4 ? 4 : 2);
};

template <int W, int POLICY>
struct DirectCfg {
    static constexpr int NARR = 2 + W + (POLICY == KS_SCORE_LEAST_ALLOCATED ? 2 : 0);
    static constexpr uint32_t STAGE_BYTES = (uint32_t)NARR * TILE_N * 8u;
    static constexpr uint32_t SMEM_BYTES = 2u * STAGE_BYTES;
};

template <int W, int POLICY, bool EMIT_MASK>
__global__ void __launch_bounds__(DIRECT_THREADS)
    k_select_direct(NodeTable nt, PodView pv, OutView ov, PartialView part, uint32_t tiles_per_chunk) {
    constexpr int PW = PodsPerWarp<W>::v;
    using Cfg = DirectCfg<W, POLICY>;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ __align__(8) uint64_t full_bar[2];

    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t n_tiles_total = nt.Npad / TILE_N;
    const uint32_t tile_begin = blockIdx.y * tiles_per_chunk;
    const uint32_t tile_end = min(tile_begin + tiles_per_chunk, n_tiles_total);

    if (threadIdx.x == 0) {
        mbar_init(&full_bar[0], 1);
        mbar_init(&full_bar[1], 1);
        fence_mbar_init();
    }
    __syncthreads();

    auto issue_tile = [&](uint32_t tile, uint32_t stage) {
        // one elected thread arms the barrier with the byte count, then issues one bulk copy per SoA column
        unsigned char* dst = smem_raw + (size_t)stage * Cfg::STAGE_BYTES;
        uint64_t* bar = &full_bar[stage];
        mbar_arrive_expect_tx(bar, Cfg::STAGE_BYTES);
        const size_t off = (size_t)tile * TILE_N;
        tma_bulk_g2s(dst, nt.free_cpu + off, TILE_N * 8, bar);
        tma_bulk_g2s(dst + TILE_N * 8, nt.free_mem + off, TILE_N * 8, bar);
#pragma unroll
        for (int w = 0; w < W; w++)
            tma_bulk_g2s(dst + (2 + w) * TILE_N * 8, nt.labels + (size_t)w * nt.Npad + off, TILE_N * 8, bar);
        if (POLICY == KS_SCORE_LEAST_ALLOCATED) {
            tma_bulk_g2s(dst + (2 + W) * TILE_N * 8, nt.alloc_cpu + off, TILE_N * 8, bar);
            tma_bulk_g2s(dst + (3 + W) * TILE_N * 8, nt.alloc_mem + off, TILE_N * 8, bar);
        }
    };

    if (threadIdx.x == 0 && tile_begin < tile_end) issue_tile(tile_begin, 0);

    // this warp's pods (uniform registers)
    const uint32_t p0 = (blockIdx.x * (DIRECT_THREADS / 32) + warp) * PW;
    int64_t rc[PW], rm[PW];
    uint64_t sel[PW][W];
    int64_t best[PW];
    int32_t bidx[PW];
    uint32_t cnt[PW];
    uint32_t acc[PW];
#pragma unroll
    for (int i = 0; i < PW; i++) {
        uint32_t p = min(p0 + i, pv.P - 1);
        rc[i] = __ldg(pv.req_cpu + p);
        rm[i] = __ldg(pv.req_mem + p);
#pragma unroll
        for (int w = 0; w < W; w++) sel[i][w] = __ldg(pv.sel + (uint64_t)p * W + w);
        best[i] = INT64_MIN;
        bidx[i] = -1;
        cnt[i] = 0;
        acc[i] = 0;
    }

    for (uint32_t tile = tile_begin; tile < tile_end; tile++) {
        const uint32_t it = tile - tile_begin, stage = it & 1;
        if (threadIdx.x == 0 && tile + 1 < tile_end) issue_tile(tile + 1, stage ^ 1);
        mbar_wait(&full_bar[stage], (it >> 1) & 1);

        const unsigned char* base = smem_raw + (size_t)stage * Cfg::STAGE_BYTES;
        const int64_t* s_fc = reinterpret_cast<const int64_t*>(base);
        const int64_t* s_fm = s_fc + TILE_N;
        const uint64_t* s_lab = reinterpret_cast<const uint64_t*>(s_fm + TILE_N);
        const int64_t* s_ac = reinterpret_cast<const int64_t*>(s_lab + (size_t)W * TILE_N);
        const int64_t* s_am = s_ac + TILE_N;

#pragma unroll 2
        for (uint32_t g = 0; g < 32; g++) {
            const uint32_t ln = g * 32 + lane;
            const int64_t fc = s_fc[ln], fm = s_fm[ln];
            uint64_t lab[W];
#pragma unroll
            for (int w = 0; w < W; w++) lab[w] = s_lab[w * TILE_N + ln];
            const int32_t node = (int32_t)(tile * TILE_N + ln);
            const bool real = (uint32_t)node < nt.N; // padding sentinels are never feasible
            int64_t key_n = 0, ac = 0, am = 0;
            if (POLICY == KS_SCORE_LEFTOVER) {
                key_n = leftover_prio(fc, fm); // the pod part is constant
            } else {
                ac = s_ac[ln];
                am = s_am[ln];
            }
#pragma unroll
            for (int i = 0; i < PW; i++) {
                const bool fit = (rc[i] <= fc) & (rm[i] <= fm);
                uint64_t miss = 0;
#pragma unroll
                for (int w = 0; w < W; w++) miss |= sel[i][w] & ~lab[w];
                const bool ok = fit && (miss == 0) && real;
                const uint32_t b = __ballot_sync(0xffffffffu, ok);
                cnt[i] += __popc(b);
                if (EMIT_MASK) acc[i] = (lane == g) ? b : acc[i];
                // ascending node per lane: strict '>' is argmax_better here, and cheaper
                if (POLICY == KS_SCORE_LEFTOVER) {
                    if (ok && key_n > best[i]) {
                        best[i] = key_n;
                        bidx[i] = node;
                    }
                } else {
                    if (ok) {
                        const int64_t s = least_alloc_score(fc, fm, ac, am, rc[i], rm[i]);
                        if (s > best[i]) {
                            best[i] = s;
                            bidx[i] = node;
                        }
                    }
                }
            }
        }
        if (EMIT_MASK) {
            const uint32_t word = tile * 32 + lane; // 32 words per 1024-node tile
            if (word < ov.mask_valid_words) {
#pragma unroll
                for (int i = 0; i < PW; i++)
                    if (p0 + i < pv.P) ov.mask[(uint64_t)(p0 + i) * ov.mask_row_words + word] = acc[i];
            }
        }
        __syncthreads(); // everyone is done with `stage` before it is refilled two iterations later
    }

#pragma unroll
    for (int i = 0; i < PW; i++) {
        const Candidate w = warp_argmax(best[i], bidx[i]);
        if (lane == 0 && p0 + i < pv.P) {
            const uint32_t p = p0 + i;
            if (gridDim.y == 1) {
                const int64_t s = w.idx >= 0 ? key_to_score(POLICY, w.key, rc[i], rm[i]) : 0;
                if (ov.node_idx) ov.node_idx[p] = w.idx;
                if (ov.score) ov.score[p] = s;
                if (ov.cnt) ov.cnt[p] = cnt[i];
            } else {
                const uint64_t o = (uint64_t)blockIdx.y * pv.P + p;
                part.key[o] = w.key;
                part.idx[o] = w.idx;
                part.cnt[o] = cnt[i];
            }
        }
    }
}

// combine partials of node chunks
template <int POLICY>
__global__ void k_select_combine(PodView pv, OutView ov, PartialView part, uint32_t n_chunks) {
    uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= pv.P) return;
    int64_t k = INT64_MIN;
    int32_t ix = -1;
    uint32_t c = 0;
    for (uint32_t ch = 0; ch < n_chunks; ch++) {
        const uint64_t o = (uint64_t)ch * pv.P + p;
        c += part.cnt[o];
        int32_t oi = part.idx[o];
        int64_t ok_ = part.key[o];
        if (argmax_better(ok_, oi, k, ix)) {
            k = ok_;
            ix = oi;
        }
    }
    const int64_t s = ix >= 0 ? key_to_score(POLICY, k, pv.req_cpu[p], pv.req_mem[p]) : 0;
    if (ov.node_idx) ov.node_idx[p] = ix;
    if (ov.score) ov.score[p] = s;
    if (ov.cnt) ov.cnt[p] = c;
}

template <int W, int POLICY, bool EMIT>
static cudaError_t launch_direct_t(const SelectLaunch& L, const PartialView& part, uint32_t n_chunks,
                                   uint32_t tiles_per_chunk) {
    using Cfg = DirectCfg<W, POLICY>;
    constexpr int PW = PodsPerWarp<W>::v;
    auto kern = k_select_direct<W, POLICY, EMIT>;
    cudaError_t e;
    const uint32_t pods_per_cta = (DIRECT_THREADS / 32) * PW;
    dim3 grid((L.pv.P + pods_per_cta - 1) / pods_per_cta, n_chunks);
    kern<<<grid, DIRECT_THREADS, Cfg::SMEM_BYTES, L.stream>>>(L.nt, L.pv, L.ov, part, tiles_per_chunk);
    g_launches++;
    e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    if (n_chunks > 1) {
        k_select_combine<POLICY><<<(L.pv.P + 255) / 256, 256, 0, L.stream>>>(L.pv, L.ov, part, n_chunks);
        g_launches++;
        e = cudaGetLastError();
    }
    return e;
}

template <int W>
static cudaError_t launch_direct_w(const SelectLaunch& L, const PartialView& part, uint32_t n_chunks,
                                   uint32_t tiles_per_chunk) {
    const bool emit = L.ov.mask != nullptr;
    if (L.policy == KS_SCORE_LEFTOVER)
        return emit ? launch_direct_t<W, KS_SCORE_LEFTOVER, true>(L, part, n_chunks, tiles_per_chunk)
                    : launch_direct_t<W, KS_SCORE_LEFTOVER, false>(L, part, n_chunks, tiles_per_chunk);
    return emit ? launch_direct_t<W, KS_SCORE_LEAST_ALLOCATED, true>(L, part, n_chunks, tiles_per_chunk)
                : launch_direct_t<W, KS_SCORE_LEAST_ALLOCATED, false>(L, part, n_chunks, tiles_per_chunk);
}

template <int W>
static cudaError_t prepare_w() {
    cudaError_t e;
#define KS_SET(P_, M_)                                                                                            \
    if ((e = cudaFuncSetAttribute(k_select_direct<W, P_, M_>, cudaFuncAttributeMaxDynamicSharedMemorySize,        \
                                  (int)DirectCfg<W, P_>::SMEM_BYTES)) != cudaSuccess)                             \
        return e;
    KS_SET(KS_SCORE_LEFTOVER, true)
    KS_SET(KS_SCORE_LEFTOVER, false)
    KS_SET(KS_SCORE_LEAST_ALLOCATED, true)
    KS_SET(KS_SCORE_LEAST_ALLOCATED, false)
#undef KS_SET
    return cudaSuccess;
}

// opt-in shared memory sizes, once per label width (must not run inside a stream capture)
cudaError_t prepare_select_direct(uint32_t W) {
    static bool done[9] = {false, false, false, false, false, false, false, false, false};
    if (W > 8) return cudaErrorInvalidValue;
    if (done[W]) return cudaSuccess;
    cudaError_t e = cudaErrorInvalidValue;
    switch (W) {
        case 1: e = prepare_w<1>(); break;
        case 2: e = prepare_w<2>(); break;
        case 4: e = prepare_w<4>(); break;
        case 8: e = prepare_w<8>(); break;
        default: break;
    }
    if (e == cudaSuccess) done[W] = true;
    return e;
}

uint32_t direct_pods_per_cta(uint32_t W) {
    switch (W) {
        case 1: return (DIRECT_THREADS / 32) * PodsPerWarp<1>::v;
        case 2: return (DIRECT_THREADS / 32) * PodsPerWarp<2>::v;
        case 4: return (DIRECT_THREADS / 32) * PodsPerWarp<4>::v;
        default: return (DIRECT_THREADS / 32) * PodsPerWarp<8>::v;
    }
}

cudaError_t launch_select_direct(const SelectLaunch& L, const PartialView& part, uint32_t n_chunks,
                                 uint32_t tiles_per_chunk) {
    switch (L.nt.W) {
        case 1: return launch_direct_w<1>(L, part, n_chunks, tiles_per_chunk);
        case 2: return launch_direct_w<2>(L, part, n_chunks, tiles_per_chunk);
        case 4: return launch_direct_w<4>(L, part, n_chunks, tiles_per_chunk);
        case 8: return launch_direct_w<8>(L, part, n_chunks, tiles_per_chunk);
        default: return cudaErrorInvalidValue;
    }
}

} // namespace ks
