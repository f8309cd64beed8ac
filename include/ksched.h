/* ksched.h — C ABI of the B200 scheduling core (libksched.so).
 *
 * Drop-in boundary for the hot path of acrlabs/kube-scheduler-rs-reference.  The reference is a binary
 * crate with no FFI; the three in-crate functions this library replaces are (paths relative to
 * /root/reference):
 *   check_node_validity(&Pod,&Node,&Context) -> Result<(),InvalidNodeReason>   src/predicates.rs:63-77
 *   select_node_for_pod(&Pod,&Context) -> Option<Node>                         src/main.rs:51-71
 *   Context{client,node_store} (node cache + per-cell LIST of bound pods)      src/util.rs:12-15,
 *                                                                              src/predicates.rs:21-38
 * A Rust host would bind these entry points with an `extern "C"` block (INTEGRATION.md shows it);
 * signatures use only plain pointers, sizes and opaque handles.  No torch / C++ types cross the ABI.
 *
 * Units: cpu = int64 millicores, memory = int64 bytes, labels = W x uint64 bit columns per row
 * (bit set on a node = node carries that (key,value) pair; bit set on a pod = selector requires it).
 * Cell semantics (bit-exact with oracle/oracle.c):
 *   fit   = req_cpu <= free_cpu && req_mem <= free_mem          (src/predicates.rs:42, non-strict)
 *   match = for all w: (sel[w] & ~labels[w]) == 0               (src/predicates.rs:45-61)
 *   code  = !fit ? 1 : !match ? 2 : 0                           (src/predicates.rs:68-76, fit first)
 * All functions return KS_OK (0) or a negative KS_ERR_*; nothing aborts or throws across the ABI
 * (the reference panics on malformed data, src/predicates.rs:29,31,36).  ks_last_error() returns a
 * thread-local description of the most recent failure on the calling thread.
 */
#ifndef KSCHED_H
#define KSCHED_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define KS_OK 0
#define KS_ERR_INVALID (-1)
#define KS_ERR_CUDA (-2)
#define KS_ERR_PARSE (-3)
#define KS_ERR_NOMEM (-4)
#define KS_ERR_RANGE (-5)
#define KS_ERR_INEXACT (-6)
#define KS_ERR_MISSING (-7)
#define KS_ERR_NO_DEVICE (-8)

/* cell codes = Ok(()) / InvalidNodeReason (src/predicates.rs:14-18) */
#define KS_CELL_OK 0
#define KS_CELL_NOT_ENOUGH_RESOURCES 1
#define KS_CELL_NODE_SELECTOR_MISMATCH 2

/* score policies (spec extension — the reference has no score; DESIGN.md "Score") */
#define KS_SCORE_LEFTOVER 0        /* (free_cpu-req_cpu)*2^22 + (free_mem-req_mem); separable => static node order */
#define KS_SCORE_LEAST_ALLOCATED 1 /* ((free_cpu-req_cpu)*100/alloc_cpu + (free_mem-req_mem)*100/alloc_mem)/2, floor */

/* where caller-owned buffers live */
#define KS_MEM_HOST 0
#define KS_MEM_DEVICE 1

/* ks_select flags */
#define KS_SELECT_AUTO 0u
#define KS_SELECT_FORCE_DIRECT 1u  /* per-cell kernel (any policy) */
#define KS_SELECT_FORCE_BITPAR 2u  /* bit-parallel kernel (any policy) */
#define KS_SELECT_TIMING 4u        /* record CUDA events around each kernel; read with ks_last_timings */
#define KS_SELECT_NO_GRAPH 8u      /* repeated calls whose buffers are device or pinned host memory are replayed from a
                                      cached CUDA graph; this disables it */

/* value limits enforced on inputs so that scores and sums stay inside int64 */
#define KS_MAX_CPU_MILLI ((int64_t)1 << 36)
#define KS_MAX_MEM_BYTES ((int64_t)1 << 55)
#define KS_MAX_LABEL_WORDS 8u

typedef struct ks_snapshot ks_snapshot; /* replaces Context.node_store + the LIST, src/util.rs:12-15 */

typedef struct ks_pods { /* SoA view of P pending pods (what total_pod_resources + node_selector pack to) */
    uint64_t n;
    const int64_t* req_cpu;  /* [n] millicores   (src/util.rs:54-75 per pod) */
    const int64_t* req_mem;  /* [n] bytes */
    const uint64_t* sel;     /* [n*W] required label bits (all zero = no selector) */
    int32_t mem_space;       /* KS_MEM_HOST or KS_MEM_DEVICE for the three arrays above */
} ks_pods;

/* ---- multi-GPU exchange of the bindings (SURVEY.md section 8e; one process per GPU, pods sharded) ----
 * The reference has no multi-process story; north_star asks for ONE all-gather of the per-pod bindings.  Here the
 * all-gather is fused into the argmax kernels: every binding is stored into the local output AND into every peer's
 * gather buffer through peer-mapped (CUDA IPC) pointers over NVLink, then one flag per (source, destination) pair is
 * released; ks_select ends with a wait on this rank's flags, so when the call's stream work is done the gather
 * buffer holds the bindings of every rank.  No collective library call is on the data path.
 * All pointers are DEVICE pointers valid in the calling process (peer_* ones were opened with ks_ipc_open). */
#define KS_MAX_PEERS 15u
typedef struct ks_exchange {
    uint32_t world, rank;                 /* ranks taking part, this rank */
    uint32_t n_peers;                     /* = world - 1 */
    int32_t* peer_node_idx[KS_MAX_PEERS]; /* where THIS rank's node_idx[0..n) goes in peer k's gather buffer */
    int64_t* peer_score[KS_MAX_PEERS];    /* same for score */
    uint32_t* peer_flag[KS_MAX_PEERS];    /* peer k's arrival flag for THIS rank */
    uint32_t* local_flags;                /* this rank's flags [world]; entry r is written by rank r */
    uint32_t* local_state;                /* this rank's private words [16], zeroed, 8-byte aligned: [0] step sequence
                                             number, [1] CTA counter, [2..11] five 64-bit %globaltimer stamps (ns) of
                                             the last step: first argmax CTA, flags published, wait started, wait done,
                                             second argmax kernel started */
} ks_exchange;

typedef struct ks_bindings { /* outputs; any pointer may be NULL to skip that output */
    int32_t* node_idx;       /* [n] argmax-score feasible node, ties -> lowest index, -1 = NoNodeFound */
    int64_t* score;          /* [n] score of node_idx (0 when -1) */
    uint32_t* feasible_cnt;  /* [n] number of feasible nodes */
    int32_t mem_space;       /* space of the three arrays above */
    uint8_t* mask;           /* [n rows] feasible bit-mask, bit (n%8) of byte n/8 of the row */
    uint64_t mask_row_bytes; /* row pitch; multiple of 32, >= ks_mask_row_bytes(N); ks_mask_row_bytes_aligned(N) is fastest */
    int32_t mask_space;      /* space of mask (may differ: keep a 6 GB mask in HBM, bindings on host) */
    void* bindings_ready_event; /* optional cudaEvent_t (NULL = none), device-space outputs only: recorded as soon as
                                   node_idx and score are final - on the bit-parallel path that is well before the
                                   mask/count pass ends, so a collective over the bindings can overlap it */
    const ks_exchange* exchange; /* optional (NULL = none), device-space outputs only: fused all-gather, see above */
} ks_bindings;

const char* ks_last_error(void);
int ks_version(void);
int ks_device_count(void);           /* number of CUDA devices visible; 0 when none */
uint64_t ks_launch_count(void);      /* kernels launched by this library since load */
uint64_t ks_mask_row_bytes(uint32_t n_nodes); /* 32 * ceil(n_nodes/256): the smallest legal row pitch */
/* 256 * ceil(n_nodes/2048): the recommended pitch for a device-space mask.  The mask kernel writes one 256-byte block
 * per (pod, 2048-node column block); with this pitch (and a 256-byte-aligned base) every block is whole and aligned,
 * which the memory system of a B200 rewards with ~1.35x the store bandwidth of straddling blocks.  Bytes of a row
 * beyond ks_mask_row_bytes(n_nodes) carry no information: up to the aligned size the bit-parallel path writes them
 * as zeros (whole 32-byte tiles that fit the pitch), the per-cell path leaves them untouched. */
uint64_t ks_mask_row_bytes_aligned(uint32_t n_nodes);

/* ---- snapshot: device-resident node table (replaces node_store.state(), src/main.rs:56) ---- */
int ks_snapshot_create(int device, ks_snapshot** out);
void ks_snapshot_destroy(ks_snapshot* s);
/* host arrays; labels = [n_nodes*label_words]; resets bound load (free = alloc). */
int ks_snapshot_set_nodes(ks_snapshot* s, uint32_t n_nodes, uint32_t label_words, const int64_t* alloc_cpu,
                          const int64_t* alloc_mem, const uint64_t* labels);
/* K0: free[n] = alloc[n] - sum over bound pods on n (src/predicates.rs:27-38).  host arrays. */
int ks_snapshot_set_bound(ks_snapshot* s, uint64_t n_bound, const int32_t* node_idx, const int64_t* req_cpu,
                          const int64_t* req_mem);
/* incremental: one more pod bound to node_idx (what the next LIST would show after src/main.rs:103) */
int ks_snapshot_apply_bind(ks_snapshot* s, int32_t node_idx, int64_t req_cpu, int64_t req_mem);
int ks_snapshot_get_free(ks_snapshot* s, int64_t* free_cpu, int64_t* free_mem); /* D2H, [n_nodes] each */
uint32_t ks_snapshot_num_nodes(const ks_snapshot* s);
uint32_t ks_snapshot_label_words(const ks_snapshot* s);

/* ---- device memory that other processes of the node can map (CUDA IPC), for ks_exchange ----
 * ks_ipc_alloc: cudaMalloc + zero fill on `device`; out_handle receives the 64-byte cudaIpcMemHandle_t to send to the
 * peers (any byte transport: torch.distributed, MPI, a file).  ks_ipc_open maps a peer's allocation into this process
 * (peer access between the two GPUs is enabled by the runtime).  ks_ipc_close / ks_ipc_free undo them. */
/* after a run of ks_select calls with an exchange: synchronises the device and reports whether any wait timed out */
int ks_exchange_check(ks_snapshot* s);
int ks_ipc_alloc(int device, uint64_t bytes, void** out_ptr, uint8_t out_handle[64]);
int ks_ipc_open(int device, const uint8_t handle[64], void** out_ptr);
int ks_ipc_close(int device, void* ptr);
int ks_ipc_free(int device, void* ptr);
/* store-only bandwidth of the device: best of `iters` passes of a plain coalesced 256-bit-store fill over dev_buf
 * (bytes >= 1 MiB, 32-byte aligned; its contents are overwritten).  MEASURED_PEAKS-style HBM peaks are copies
 * (read + write bytes); a kernel that only writes - the feasible-mask pass - is bounded by this figure instead. */
int ks_measure_write_bandwidth(int device, void* dev_buf, uint64_t bytes, int iters, double* out_gbs);
/* synchronising device-to-host copy of `bytes` bytes (reading a gather buffer allocated with ks_ipc_alloc) */
int ks_device_read(int device, const void* dev_ptr, void* host_ptr, uint64_t bytes);

/* ---- per-cell entry = check_node_validity (src/predicates.rs:63-77) ---- */
int ks_check_cell(ks_snapshot* s, int64_t req_cpu, int64_t req_mem, const uint64_t* sel, uint32_t node_idx);
/* K1: all P*N reason codes, out_codes[p*N+n] in host memory (small problems / parity tests) */
int ks_check_cells(ks_snapshot* s, const ks_pods* pods, uint8_t* out_codes);

/* ---- per-pod batched entry = select_node_for_pod over P pods ("predicates::run") ---- */
int ks_select(ks_snapshot* s, const ks_pods* pods, int policy, uint32_t flags, ks_bindings* out,
              void* cuda_stream /* cudaStream_t or NULL = library stream; call returns after completion
                                   for host-space outputs, after enqueue for all-device outputs */);
/* milliseconds of the kernels of the last KS_SELECT_TIMING call on this snapshot:
 * ms[0]=dominant mask/score kernel, ms[1]=argmax scan / combine, ms[2]=total enqueue-to-done. */
int ks_last_timings(ks_snapshot* s, float ms[3]);
/* name of the dominant kernel path the last ks_select used: "direct" or "bitpar" */
const char* ks_last_path(const ks_snapshot* s);
/* Timeline of the last bit-parallel ks_select on this snapshot, from %globaltimer stamps written by the kernels
 * themselves (the streams of a step overlap, which per-kernel profilers serialise).  Only when the process runs with
 * KS_TRACE=1 in its environment (else KS_ERR_INVALID); synchronises the device.  out_ns[k], nanoseconds of the
 * device clock, 0 = kernel did not run:  0/1 pod-rank kernel first CTA start / last CTA end, 2/3 first argmax kernel,
 * 4/5 second argmax kernel, 6/7 mask kernel, 8 end of the mask CTA that finished first; 9..15 reserved (0). */
int ks_last_trace(ks_snapshot* s, uint64_t out_ns[16]);

/* ---- streaming reconcile (BASELINE.json config C5): micro-batches against the resident snapshot ----
 * The reference re-LISTs bound pods for every cell (src/predicates.rs:34), so a pod always sees earlier binds.
 * A batched pass sees one snapshot, so two pods of a batch may claim the same capacity.  K3 resolves that:
 * claims are taken per node in arrival (array) order; a claim is accepted iff its request still fits what is
 * left on the node, and then decrements it.  Capacity never goes negative through this path.
 *
 * ks_snapshot_commit_claims: host arrays; claim i = pod i wants node claim_node[i] (-1 = no claim).
 *   out_accepted[i] = 1/0.  Accepted requests are subtracted from free[] on the device (same effect as
 *   ks_snapshot_apply_bind per accepted claim).  Every replica that commits the same claim list in the same
 *   order ends with the same free[] (multi-GPU streaming: all-gather the claims, commit everywhere).
 * ks_stream_bind: the full micro-batch loop on one GPU — select (per-cell kernel, any policy) for the pending
 *   pods, commit, re-select the losers against the updated free[], until every pod is bound or has no feasible
 *   node.  out_node_idx[i] = bound node or -1 (= ReconcileError::NoNodeFound, src/main.rs:116-118). */
int ks_snapshot_commit_claims(ks_snapshot* s, uint64_t n_claims, const int32_t* claim_node, const int64_t* req_cpu,
                              const int64_t* req_mem, uint8_t* out_accepted);
int ks_stream_bind(ks_snapshot* s, const ks_pods* pods /* host space */, int policy, int32_t* out_node_idx,
                   int64_t* out_score, uint32_t* out_rounds);

/* ---- asynchronous streaming surface = the reference's Controller queue (src/main.rs:73, :141-148) ----
 * The reference runs reconcile() for many pods concurrently from a work queue.  ks_stream is that queue in front of
 * one snapshot: ks_stream_submit appends pending (unbound) pods and returns at once; a dispatcher thread owned by the
 * library drains everything that has arrived (up to max_batch <= 1024 pods, arrival order) into ONE micro-batch
 * (ks_stream_bind: device-side round loop with capacity commit) and publishes the results; ks_stream_poll collects
 * finished pods without blocking.  Results carry the caller's ticket; node -1 = ReconcileError::NoNodeFound
 * (src/main.rs:116-118).  Pods with spec.nodeName set must be filtered out before submission (src/main.rs:74-76).
 * While a stream is open its snapshot must not be mutated by other calls (same rule as the reference's node store
 * being written only by its reflector). */
typedef struct ks_stream ks_stream;
int ks_stream_open(ks_snapshot* s, int policy, uint32_t max_batch, ks_stream** out);
int ks_stream_submit(ks_stream* q, uint64_t n, const int64_t* req_cpu, const int64_t* req_mem, const uint64_t* sel /* [n*W] */,
                     const uint64_t* tickets /* [n] caller ids, returned by poll */);
/* up to `max` finished pods; *out_n = how many were written (0 = nothing finished yet); never blocks */
int ks_stream_poll(ks_stream* q, uint64_t max, uint64_t* out_ticket, int32_t* out_node_idx, int64_t* out_score, uint64_t* out_n);
int ks_stream_flush(ks_stream* q);  /* blocks until every pod submitted so far has a result waiting in poll */
int ks_stream_stats(ks_stream* q, uint64_t* batches, uint64_t* rounds, uint64_t* max_batch_seen);
void ks_stream_close(ks_stream* q); /* stops the dispatcher; unpolled results are dropped */

/* ---- the reference's own selection policy, seeded (src/main.rs:49-71; ATTEMPTS = 5 at :49) ----
 * For every pod: up to `attempts` draws, uniform with replacement over the snapshot's nodes (:56-57); the first
 * draw whose cell is KS_CELL_OK wins (:61-66); none -> -1 (= None -> ReconcileError::NoNodeFound, :70, :116-118)
 * even when a feasible node exists.  The reference draws from thread_rng; here draw k of pod p is
 * splitmix64 step k of a stream whose state starts at KS_SAMPLING_STREAM(seed, p), node = draw % N, so a run is
 * reproducible and replicas agree.  An empty snapshot wastes every attempt (:56,60): -1, 0 cells.
 * Host output arrays; all but out_node_idx may be NULL:
 *   out_node_idx[P]; out_attempts[P] = cells evaluated; out_draw_node[P*attempts] = node of each draw (-1 = not
 *   made); out_draw_code[P*attempts] = that cell's code, i.e. the InvalidNodeReason the reference logs at :62
 *   (0xff = not made).  first_pod_index offsets p in the stream id (pod i of this call is stream
 *   first_pod_index + i), so a sharded or chunked caller reproduces the single-call result. */
#define KS_REFERENCE_ATTEMPTS 5u
#define KS_SAMPLING_STREAM(seed, p) ((uint64_t)(seed) ^ (((uint64_t)(p) + 1ull) * 0xD1B54A32D192ED03ull))
int ks_select_sampling(ks_snapshot* s, const ks_pods* pods, uint32_t attempts, uint64_t seed, uint64_t first_pod_index,
                       int32_t* out_node_idx, uint32_t* out_attempts, int32_t* out_draw_node, uint8_t* out_draw_code);

#ifdef __cplusplus
}
#endif
#endif /* KSCHED_H */
