// ks_stream.cu — K3: in-batch conflict resolution + capacity commit for streaming reconcile (config C5).
// Mirrors what the reference gets from re-LISTing bound pods per cell (/root/reference/src/predicates.rs:34-38):
// a later pod of the batch sees the capacity taken by earlier pods of the same batch.
#include "ks_internal.cuh"
#include "ks_launch.h"

#include <cooperative_groups.h>
namespace cg = cooperative_groups;

namespace ks {

constexpr int STREAM_MAX = 4096; // claims per launch (one CTA sorts them in shared memory)
constexpr uint32_t RESOLVE_THREADS = 1024;

// One CTA resolves the caller's claims (resolve_claims); a claim on a node outside [0, N) is rejected.
__global__ void __launch_bounds__(RESOLVE_THREADS)
    k_stream_resolve(int64_t* __restrict__ free_cpu, int64_t* __restrict__ free_mem, const int32_t* __restrict__ claim_node,
                     const int64_t* __restrict__ req_cpu, const int64_t* __restrict__ req_mem, uint32_t n, uint32_t N,
                     uint8_t* __restrict__ accepted) {
    __shared__ unsigned long long key[STREAM_MAX];
    for (uint32_t i = threadIdx.x; i < n; i += RESOLVE_THREADS) {
        const int32_t nd = claim_node[i];
        const bool valid = nd >= 0 && (uint32_t)nd < N;
        if (!valid) accepted[i] = 0;
        key[i] = valid ? ((unsigned long long)(uint32_t)nd << 32) | i : ~0ull;
    }
    resolve_claims<RESOLVE_THREADS>(
        key, n, free_cpu, free_mem, [&](uint32_t c) { return make_longlong2(req_cpu[c], req_mem[c]); },
        [&](uint32_t c, bool ok) { accepted[c] = ok; });
}

cudaError_t launch_stream_resolve(int64_t* free_cpu, int64_t* free_mem, const int32_t* claim_node, const int64_t* req_cpu,
                                  const int64_t* req_mem, uint32_t n, uint32_t N, uint8_t* accepted, cudaStream_t st) {
    if (n == 0) return cudaSuccess;
    if (n > STREAM_MAX) return cudaErrorInvalidValue;
    k_stream_resolve<<<1, RESOLVE_THREADS, 0, st>>>(free_cpu, free_mem, claim_node, req_cpu, req_mem, n, N, accepted);
    g_launches++;
    return cudaGetLastError();
}

uint32_t stream_max_claims() { return STREAM_MAX; }

// ------------------------------------------------------------------------------------------------ device-side loop
// k_stream_batch: the whole micro-batch loop of ks_stream_bind in ONE cooperative launch (no host round trip per
// round).  Per round, exactly as the host loop / the oracle (orc_stream_bind_packed):
//   A  every CTA scans its slice of the node table for every pending pod (one warp per pod, lanes over nodes):
//      feasible (predicates.rs:42,45-61) -> policy key -> warp argmax (ties -> lowest node index) -> partial[pod][cta]
//   B  CTA 0 reduces the partials to one claim per pod, resolves the claims per node in arrival order against what
//      is left (resolve_claims, as k_stream_resolve), commits the accepted requests to free[], writes the bindings and
//      compacts the losers (order preserved) into the next round's pending list
// separated by grid-wide barriers.  Batches of up to STREAM_BATCH_MAX pods.
constexpr uint32_t SB_THREADS = 256;

template <int W>
__global__ void __launch_bounds__(SB_THREADS)
    k_stream_batch(uint32_t N, uint32_t Npad, const int64_t* __restrict__ alloc_cpu, const int64_t* __restrict__ alloc_mem,
                   const uint64_t* __restrict__ labels, int64_t* free_cpu, int64_t* free_mem, int policy, uint32_t m,
                   const int64_t* __restrict__ req_cpu, const int64_t* __restrict__ req_mem, const uint64_t* __restrict__ sel,
                   int64_t* pkey, int32_t* pidx, uint32_t* pend, uint32_t* ctl, int32_t* out_idx, int64_t* out_score,
                   uint32_t max_rounds) {
    cg::grid_group grid = cg::this_grid();
    __shared__ unsigned long long s_key[STREAM_BATCH_MAX];
    __shared__ int64_t s_ckey[STREAM_BATCH_MAX];
    __shared__ int32_t s_claim[STREAM_BATCH_MAX];
    __shared__ uint8_t s_acc[STREAM_BATCH_MAX];
    __shared__ uint32_t s_scan[SB_THREADS];
    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, G = gridDim.x;
    const uint32_t chunk = (N + G - 1) / G, n0 = min(N, blockIdx.x * chunk), n1 = min(N, n0 + chunk);
    if (blockIdx.x == 0) {
        for (uint32_t i = tid; i < m; i += SB_THREADS) {
            pend[i] = i;
            out_idx[i] = -1; // NoNodeFound until bound (src/main.rs:116-118)
            out_score[i] = 0;
        }
        if (tid == 0) {
            ctl[0] = m;
            ctl[1] = 0;
        }
        __threadfence();
    }
    grid.sync();
    uint32_t cur = 0;
    for (uint32_t round = 0;; round++) {
        const uint32_t cnt = *reinterpret_cast<volatile uint32_t*>(ctl);
        if (cnt == 0 || round > max_rounds) break; // grid-uniform
        const uint32_t* pl = pend + cur * STREAM_BATCH_MAX;
        // ---- A: partial argmax over this CTA's node slice ----
        for (uint32_t k = warp; k < cnt; k += SB_THREADS / 32) {
            const uint32_t p = __ldcg(pl + k);
            const int64_t rc = req_cpu[p], rm = req_mem[p];
            uint64_t sw[W];
#pragma unroll
            for (int w = 0; w < W; w++) sw[w] = sel[(size_t)p * W + w];
            int64_t best = INT64_MIN;
            int32_t bidx = -1;
            for (uint32_t n = n0 + lane; n < n1; n += 32) {
                const int64_t fc = __ldcg(free_cpu + n), fm = __ldcg(free_mem + n); // free[] changes between rounds
                uint64_t miss = 0;
#pragma unroll
                for (int w = 0; w < W; w++) miss |= sw[w] & ~labels[(size_t)w * Npad + n];
                if (rc <= fc && rm <= fm && miss == 0) {
                    const int64_t key = policy == KS_SCORE_LEFTOVER
                                            ? leftover_prio(fc, fm)
                                            : least_alloc_score(fc, fm, alloc_cpu[n], alloc_mem[n], rc, rm);
                    if (key > best) { // ascending n per lane: strict '>' is argmax_better here, and cheaper
                        best = key;
                        bidx = (int32_t)n;
                    }
                }
            }
            const Candidate w = warp_argmax(best, bidx);
            if (lane == 0) {
                pkey[(size_t)k * G + blockIdx.x] = w.key;
                pidx[(size_t)k * G + blockIdx.x] = w.idx;
            }
        }
        __threadfence();
        grid.sync();
        // ---- B: CTA 0 reduces, resolves, commits, compacts ----
        if (blockIdx.x == 0) {
            for (uint32_t k = warp; k < cnt; k += SB_THREADS / 32) {
                int64_t best = INT64_MIN;
                int32_t bidx = -1;
                for (uint32_t c = lane; c < G; c += 32) { // ascending CTA = ascending node range
                    const int64_t ok_ = __ldcg(pkey + (size_t)k * G + c);
                    const int32_t oi = __ldcg(pidx + (size_t)k * G + c);
                    if (argmax_better(ok_, oi, best, bidx)) {
                        best = ok_;
                        bidx = oi;
                    }
                }
                const Candidate w = warp_argmax(best, bidx);
                if (lane == 0) {
                    s_claim[k] = w.idx;
                    s_ckey[k] = w.key;
                }
            }
            __syncthreads();
            // claims per node in arrival (batch) order
            for (uint32_t i = tid; i < cnt; i += SB_THREADS) {
                s_acc[i] = 0;
                s_key[i] = s_claim[i] >= 0 ? ((unsigned long long)(uint32_t)s_claim[i] << 32) | i : ~0ull;
            }
            resolve_claims<SB_THREADS>(
                s_key, cnt, free_cpu, free_mem,
                [&](uint32_t k) {
                    const uint32_t p = __ldcg(pl + k);
                    return make_longlong2(req_cpu[p], req_mem[p]);
                },
                [&](uint32_t k, bool ok) { s_acc[k] = ok; });
            __syncthreads();
            // bindings of the winners; losers keep their order in the next pending list
            uint32_t* nl = pend + (cur ^ 1u) * STREAM_BATCH_MAX;
            constexpr uint32_t PER = STREAM_BATCH_MAX / SB_THREADS;
            uint32_t loser[PER], n_loser = 0;
#pragma unroll
            for (uint32_t e = 0; e < PER; e++) {
                const uint32_t k = tid * PER + e;
                loser[e] = 0;
                if (k < cnt && s_claim[k] >= 0) {
                    const uint32_t p = __ldcg(pl + k);
                    if (s_acc[k]) {
                        out_idx[p] = s_claim[k];
                        out_score[p] = key_to_score(policy, s_ckey[k], req_cpu[p], req_mem[p]);
                    } else {
                        loser[e] = 1;
                        n_loser++;
                    }
                }
            }
            s_scan[tid] = n_loser;
            __syncthreads();
            for (uint32_t off = 1; off < SB_THREADS; off <<= 1) { // inclusive scan (Hillis-Steele, 256 entries)
                const uint32_t v = tid >= off ? s_scan[tid - off] : 0;
                __syncthreads();
                s_scan[tid] += v;
                __syncthreads();
            }
            uint32_t pos = s_scan[tid] - n_loser;
#pragma unroll
            for (uint32_t e = 0; e < PER; e++)
                if (loser[e]) nl[pos++] = __ldcg(pl + tid * PER + e);
            if (tid == SB_THREADS - 1) {
                ctl[0] = s_scan[tid];
                ctl[1] = round + 1;
            }
            __threadfence();
        }
        grid.sync();
        cur ^= 1u;
    }
}

template <int W>
static cudaError_t launch_stream_batch_w(const StreamBatchArgs& a, cudaStream_t st) {
    StreamBatchArgs b = a;
    void* args[] = {&b.N,   &b.Npad, &b.alloc_cpu, &b.alloc_mem, &b.labels, &b.free_cpu, &b.free_mem, &b.policy,    &b.m,         &b.req_cpu,
                    &b.req_mem, &b.sel,  &b.pkey,      &b.pidx,      &b.pend,   &b.ctl,      &b.out_idx,  &b.out_score, &b.max_rounds};
    cudaError_t e = cudaLaunchCooperativeKernel(reinterpret_cast<const void*>(k_stream_batch<W>), dim3(a.grid), dim3(SB_THREADS), args, 0, st);
    if (e == cudaSuccess) g_launches++;
    return e;
}

cudaError_t launch_stream_batch(const StreamBatchArgs& a, uint32_t W, cudaStream_t st) {
    switch (W) {
        case 1: return launch_stream_batch_w<1>(a, st);
        case 2: return launch_stream_batch_w<2>(a, st);
        case 4: return launch_stream_batch_w<4>(a, st);
        case 8: return launch_stream_batch_w<8>(a, st);
        default: return cudaErrorInvalidValue;
    }
}

} // namespace ks
