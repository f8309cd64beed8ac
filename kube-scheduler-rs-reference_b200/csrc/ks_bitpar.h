// ks_bitpar.h — bit-parallel fast path (ks_bitpar.cu).
//
// Idea: `req <= free` depends only on ORDER.  Nodes are ranked once per snapshot (global position of each
// node in ascending free_cpu / free_mem order); a pod's request becomes a global rank threshold (binary
// search once per pod).  For a tile of 256 nodes the feasible bits of one resource are then a row of a
// prefix table indexed by the tile-local rank of the threshold, and the tile-local rank is
//   base[bucket][tile] + popc(member[bucket][tile] & lowmask)
// (bucket = 64 consecutive global positions).  Label selectors are ANDs of per-(key,value) node columns.
// Round 2 ("rows" kernel, the default): the tile-local rank of every possible threshold is tabulated once per
// snapshot ([column block][threshold][tile] u16, read through L1/L2), the prefix tables are octet-interleaved
// (row r of the 8 tiles of a column block = one 256-byte line, conflict-free whatever the ranks are), and one pod
// takes 8 lanes = 8 tiles = 256 contiguous bytes of its mask row: ~50 instructions per 256 cells.
// KS_SCORE_LEFTOVER is separable (node part - pod part), so argmax-score is the first
// feasible node in a static priority order: a short early-exit scan per pod (k_first_fit).
#pragma once
#include "ks_internal.cuh"

namespace ks {

constexpr int BP_TILE = 256;          // nodes per tile = 8 mask words = one 32-byte row
constexpr int BP_ROWS = BP_TILE + 1;  // prefix-table rows per tile and resource (local rank 0..256)
constexpr int BP_TABLE_BYTES = BP_ROWS * 32;
constexpr int BP_THREADS = 1024;
constexpr int BP_SMEM_MAX = 232448;   // 227 KB opt-in limit per CTA

struct BitparLayout { // byte offsets inside one column-block blob
    uint32_t nt;       // tiles per column block
    uint32_t nb;       // buckets of 64 global positions: (N >> 6) + 1
    uint32_t ncb;      // column blocks
    uint32_t off_baseC, off_membC, off_baseM, off_membM, off_tabC, off_tabM, off_pairs;
    uint32_t pstride;  // bytes between two label-pair columns
    uint32_t blob_bytes;
};

// "rows" format: column block = 8 tiles (2048 nodes).  One blob per column block:
//   tabC [257 rows][256 B], tabM [257 rows][256 B], pairs [64*W bits][256 B]
// and every 256-byte line is [half 0 of tiles 0..7 | half 1 of tiles 0..7] (16 B each): lane t of an 8-lane
// shared-memory phase reads granule t of its own row -> 8 distinct bank groups for any ranks.
constexpr uint32_t RW_TILES = 8;                            // tiles per column block
constexpr uint32_t RW_LINE = 256;                           // bytes per table row / pair column of a column block
constexpr uint32_t RW_TAB_BYTES = (uint32_t)BP_ROWS * RW_LINE; // 65792

struct RowsLayout {
    uint32_t ncb;        // column blocks
    uint32_t n_tiles;    // ceil(N / 256)
    uint32_t off_tabC, off_tabM, off_pairs; // byte offsets inside a column-block blob
    uint32_t smem_bytes; // bytes staged in shared memory (tables, + pair columns when they fit)
    uint32_t cb_stride;  // bytes between two column-block blobs in global memory
    uint32_t pairs_smem; // 1 = the pair columns are staged with the tables, 0 = read through L1/L2 (W = 8)
    uint32_t n_thr;      // thresholds per column block in the rank tables: N + 1
};

struct NodeEval;

struct BitparIndex {
    // per-snapshot index (device)
    int64_t* sortedC = nullptr;  // [N] free_cpu ascending
    int64_t* sortedM = nullptr;  // [N] free_mem ascending
    uint32_t* gposC = nullptr;   // [N] position of node n in sortedC (ties by node index)
    uint32_t* gposM = nullptr;
    int64_t* ord_prio = nullptr; // nodes in descending priority order (ties by node index), padded to a tile
    int32_t* ord_idx = nullptr;
    int64_t* splC = nullptr;     // every `spl_stride`-th element of sortedC / sortedM (<= RANK_SPLITTERS = 8192 splitters)
    int64_t* splM = nullptr;
    uint8_t* blobP = nullptr;    // one blob of layP.blob_bytes: priority order (tile k = priority ranks 256k..),
                                 // read through L1/L2 by k_first_fit_bp
    uint2* pod_ranks = nullptr;  // per-call scratch [P]
    uint32_t* tail_list = nullptr; // per-call scratch [cap_pods + 1]: pods left for k_first_fit_tail, then the count
    int64_t* ordL_s0 = nullptr;    // KS_SCORE_LEAST_ALLOCATED: score bound of every node in descending order (ties by index)
    int32_t* ordL_idx = nullptr;
    struct NodeEval* evalL = nullptr; // per slot of that order: what the exact score needs
    float4* hintL = nullptr;          // per slot of that order: single-precision score model (pre-filter of k_least_alloc)
    uint8_t* blobL = nullptr;      // flat index (layP) in that order
    unsigned long long* live = nullptr; // [KS_MAX_LABEL_WORDS] label bits carried by at least one node
    uint4* rec_s = nullptr;        // rows kernel: {threshold_cpu, threshold_mem, pod index, selector columns} per sorted pod
    uint8_t* blobR = nullptr;      // rows kernel: lay_r.ncb column-block blobs
    uint16_t* rank = nullptr;      // rows kernel: [cb][threshold g][resource][tile] = nodes of the tile at sorted positions < g
    uint32_t* tile_sorted = nullptr; // build scratch: per tile, its nodes' global positions in ascending order
    size_t cap_blobR = 0, cap_rank = 0, cap_tsorted = 0, cap_cursor = 0;
    RowsLayout lay_r{};
    uint64_t epoch = 0;            // bumped whenever a device buffer of the index is reallocated (CUDA-graph cache key)
    uint32_t* rk_hist = nullptr;   // node sample sort scratch: [3][256] bucket counts, splitters, per-node bucket / slot, lists
    int64_t* rk_spl_v = nullptr;
    uint32_t* rk_spl_i = nullptr;
    uint8_t* rk_bkt = nullptr;
    uint32_t* rk_loc = nullptr;
    uint32_t* rk_perm = nullptr;
    size_t cap_nodes = 0, cap_blobP = 0, cap_pods = 0;
    uint32_t N = 0, Nord = 0, W = 0, spl_stride = 1, n_spl = 0;
    BitparLayout layP{};
    bool valid = false;
    int sms = 0;
    cudaStream_t aux = nullptr; // the argmax kernels run here, overlapped with k_mask_rows
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    uint32_t* cursor = nullptr; // [ncb] work cursors of the mask kernel (k_mask_rows), zeroed by k_pod_ranks
    unsigned long long* trace = nullptr; // KS_TRACE=1: per-kernel %globaltimer stamps of the last select (ks_last_trace)
};
constexpr int BP_TRACE_WORDS = 16;

cudaError_t bitpar_build(BitparIndex& ix, const NodeTable& nt, int64_t* prio, cudaStream_t st);
bool bitpar_profitable(const BitparIndex& ix, uint32_t P);
cudaError_t bitpar_prepare(BitparIndex& ix, uint32_t P);
cudaError_t bitpar_select(BitparIndex& ix, SelectLaunch& L, cudaEvent_t before_mask, cudaEvent_t after_mask);
void bitpar_release(BitparIndex& ix);
// slots of ks_last_trace (include/ksched.h); cudaErrorNotSupported unless the index was created under KS_TRACE=1
cudaError_t bitpar_read_trace(const BitparIndex& ix, unsigned long long out_ns[BP_TRACE_WORDS]);

} // namespace ks
