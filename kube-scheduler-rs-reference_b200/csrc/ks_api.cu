// ks_api.cu — implementation of the C ABI declared in include/ksched.h (snapshot handle, staging,
// path selection).  Plain CUDA runtime; no torch, no oracle, no CPU fallback: every entry point that
// computes returns KS_ERR_NO_DEVICE / KS_ERR_CUDA when no B200 is present.
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <cstdlib>
#include <condition_variable>
#include <deque>
#include <mutex>
#include <thread>
#include <algorithm>
#include <type_traits>
#include <vector>

#include "ks_bitpar.h"
#include "ks_internal.cuh"
#include "ks_launch.h"

using namespace ks;

static thread_local char g_err[512] = "";

static int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

#define CU_TRY(expr)                                                                                   \
    do {                                                                                               \
        cudaError_t _e = (expr);                                                                       \
        if (_e != cudaSuccess)                                                                         \
            return fail(KS_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, \
                        __LINE__);                                                                     \
    } while (0)

// Every reallocation of a device buffer bumps this counter; it is part of the CUDA-graph cache key of ks_select, so a
// cached graph is never replayed after one of the buffers its nodes point to has moved (staging buffers grown by a
// larger call, ks_check_cells / ks_select_sampling scratch, ...).
static std::atomic<uint64_t> g_devbuf_epoch{0};

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    cudaError_t ensure(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        g_devbuf_epoch++;
        size_t want = bytes + bytes / 8 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
    template <class T>
    T* as() {
        return static_cast<T*>(p);
    }
};

enum SelectPath : uint32_t { PATH_EMPTY, PATH_DIRECT, PATH_BITPAR };

// Everything the launch sequence of a ks_select call depends on once it is captured into a CUDA graph.  The key has no
// padding, so two keys are equal exactly when memcmp says so.
struct SelectKey {
    uint64_t P;
    const void *req_cpu, *req_mem, *sel;
    const void *node_idx, *score, *feasible_cnt, *mask;
    uint64_t mask_row_bytes;
    int32_t policy, pods_space, out_space, mask_space;
    uint32_t flags, path;
    cudaStream_t stream;
    const void* ready_event;
    uint64_t version;      // ks_snapshot::version
    uint64_t devbuf_epoch; // g_devbuf_epoch
    uint64_t bitpar_epoch; // BitparIndex::epoch
    // the exchange descriptor, all zero without one: the captured kernels hold every peer pointer
    uint64_t world, rank, n_peers;
    const void *peer_node_idx[KS_MAX_PEERS], *peer_score[KS_MAX_PEERS], *peer_flag[KS_MAX_PEERS];
    const void *local_flags, *local_state;
};
static_assert(std::has_unique_object_representations_v<SelectKey>, "SelectKey is compared with memcmp: no padding");

// The launch sequence of the last ks_select that qualified, captured once and replayed while its key repeats.
struct GraphCache {
    cudaGraphExec_t exec = nullptr;
    SelectKey key{};
    bool valid = false;
    uint64_t launches = 0; // kernels inside the cached graph

    bool hit(const SelectKey& k) const { return valid && memcmp(&k, &key, sizeof(k)) == 0; }
    void reset() {
        if (exec) cudaGraphExecDestroy(exec);
        exec = nullptr;
        valid = false;
    }
    // enqueue() puts the launch sequence on `st` and returns KS_OK or an error code; on a key miss it is captured
    template <class F>
    int run(const SelectKey& k, cudaStream_t st, F&& enqueue) {
        if (!hit(k)) {
            reset();
            CU_TRY(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
            const uint64_t launches_before = g_launches.load();
            const int rc = enqueue();
            launches = g_launches.load() - launches_before; // captured, not executed yet
            g_launches -= launches;
            cudaGraph_t graph = nullptr;
            cudaError_t e = cudaStreamEndCapture(st, &graph);
            if (rc) {
                if (graph) cudaGraphDestroy(graph);
                return rc;
            }
            if (e != cudaSuccess) return fail(KS_ERR_CUDA, "stream capture failed: %s", cudaGetErrorString(e));
            e = cudaGraphInstantiate(&exec, graph, 0);
            cudaGraphDestroy(graph);
            if (e != cudaSuccess) return fail(KS_ERR_CUDA, "graph instantiate failed: %s", cudaGetErrorString(e));
            key = k;
            valid = true;
        }
        CU_TRY(cudaGraphLaunch(exec, st));
        g_launches += launches;
        return KS_OK;
    }
};

struct ks_snapshot {
    int device = 0;
    cudaStream_t stream = nullptr;
    uint32_t N = 0, Npad = 0, W = 1;
    DevBuf alloc_cpu, alloc_mem, free_cpu, free_mem, prio, labels, flag;
    DevBuf st_rc, st_rm, st_sel, st_idx, st_score, st_cnt, st_mask, st_codes, st_bnode, st_bcpu, st_bmem;
    DevBuf part_key, part_idx, part_cnt, st_samp, xflag;
    DevBuf sb_pkey, sb_pidx, sb_pend; // device-side streaming loop (k_stream_batch)
    void* h_stream = nullptr;                 // pinned staging of one streaming micro-batch (inputs and results)
    int sms = 0, coop = 0;
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
    // large host-space calls are pipelined in two pod chunks: chunk 1 is copied in on copy_stream while chunk 0 computes
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t ev_cfork = nullptr, ev_in[2] = {nullptr, nullptr};
    bool timing_valid = false;
    bool derived_dirty = true; // prio + bit-parallel index must be rebuilt before the next select
    const char* last_path = "none";
    BitparIndex bp;
    GraphCache graph;
    uint64_t version = 1; // bumped whenever device-side snapshot state or buffers change
    std::mutex mu;
};

static NodeTable node_table(ks_snapshot* s) {
    NodeTable nt;
    nt.free_cpu = s->free_cpu.as<int64_t>();
    nt.free_mem = s->free_mem.as<int64_t>();
    nt.alloc_cpu = s->alloc_cpu.as<int64_t>();
    nt.alloc_mem = s->alloc_mem.as<int64_t>();
    nt.labels = s->labels.as<uint64_t>();
    nt.N = s->N;
    nt.Npad = s->Npad;
    nt.W = s->W;
    return nt;
}

// free[] must stay inside the limits that keep scores in int64; prio[] = static node priority (KS_SCORE_LEFTOVER)
static int check_range_and_prio(ks_snapshot* s, cudaStream_t st) {
    if (s->N == 0) return KS_OK;
    CU_TRY(cudaMemsetAsync(s->flag.p, 0, sizeof(int), st));
    CU_TRY(launch_node_prio(s->free_cpu.as<int64_t>(), s->free_mem.as<int64_t>(), s->prio.as<int64_t>(), s->N, s->Npad,
                            s->flag.as<int>(), st));
    int flag = 0;
    CU_TRY(cudaMemcpyAsync(&flag, s->flag.p, sizeof(int), cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaStreamSynchronize(st));
    if (flag) return fail(KS_ERR_RANGE, "free resources of some node exceed +-2^36 millicores / +-2^55 bytes");
    return KS_OK;
}

extern "C" {

// internal hook for the host layer (host/ksh_host.cpp); not declared in include/
void ks__set_error(const char* msg) { snprintf(g_err, sizeof(g_err), "%s", msg ? msg : ""); }

const char* ks_last_error(void) { return g_err; }
int ks_version(void) { return 100; }
int ks_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}
uint64_t ks_launch_count(void) { return g_launches.load(); }
uint64_t ks_mask_row_bytes(uint32_t n_nodes) { return 32ull * ((n_nodes + 255ull) / 256ull); }
uint64_t ks_mask_row_bytes_aligned(uint32_t n_nodes) { return 256ull * ((n_nodes + 2047ull) / 2048ull); }

int ks_snapshot_create(int device, ks_snapshot** out) {
    if (!out) return fail(KS_ERR_INVALID, "out is NULL");
    *out = nullptr;
    int n = ks_device_count();
    if (n <= 0) return fail(KS_ERR_NO_DEVICE, "no CUDA device visible: libksched has no CPU fallback");
    if (device < 0 || device >= n) return fail(KS_ERR_INVALID, "device %d out of range [0,%d)", device, n);
    CU_TRY(cudaSetDevice(device));
    cudaDeviceProp prop;
    CU_TRY(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10)
        return fail(KS_ERR_NO_DEVICE, "device %d is sm_%d%d; libksched is built for sm_100a only", device, prop.major,
                    prop.minor);
    ks_snapshot* s = new (std::nothrow) ks_snapshot();
    if (!s) return fail(KS_ERR_NOMEM, "out of host memory");
    s->device = device;
    s->sms = prop.multiProcessorCount;
    s->coop = prop.cooperativeLaunch;
    cudaError_t e = cudaStreamCreateWithFlags(&s->stream, cudaStreamNonBlocking);
    for (int i = 0; i < 4 && e == cudaSuccess; i++) e = cudaEventCreate(&s->ev[i]);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&s->copy_stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s->ev_cfork, cudaEventDisableTiming);
    for (int i = 0; i < 2 && e == cudaSuccess; i++) e = cudaEventCreateWithFlags(&s->ev_in[i], cudaEventDisableTiming);
    if (e == cudaSuccess) e = s->flag.ensure(sizeof(int));
    if (e == cudaSuccess) e = s->xflag.ensure(sizeof(int));
    if (e == cudaSuccess) e = cudaMemset(s->xflag.p, 0, sizeof(int));
    if (e != cudaSuccess) {
        ks_snapshot_destroy(s);
        return fail(KS_ERR_CUDA, "snapshot init failed: %s", cudaGetErrorString(e));
    }
    *out = s;
    return KS_OK;
}

void ks_snapshot_destroy(ks_snapshot* s) {
    if (!s) return;
    cudaSetDevice(s->device);
    if (s->stream) cudaStreamSynchronize(s->stream);
    DevBuf* bufs[] = {&s->alloc_cpu, &s->alloc_mem, &s->free_cpu, &s->free_mem, &s->prio,     &s->labels,
                      &s->flag,      &s->st_rc,     &s->st_rm,    &s->st_sel,   &s->st_idx,   &s->st_score,
                      &s->st_cnt,    &s->st_mask,   &s->st_codes, &s->st_bnode, &s->st_bcpu,  &s->st_bmem,
                      &s->part_key,  &s->part_idx,  &s->part_cnt, &s->st_samp,  &s->xflag,
                      &s->sb_pkey,   &s->sb_pidx,   &s->sb_pend};
    if (s->h_stream) cudaFreeHost(s->h_stream);
    for (DevBuf* b : bufs) b->release();
    bitpar_release(s->bp);
    s->graph.reset();
    for (int i = 0; i < 4; i++)
        if (s->ev[i]) cudaEventDestroy(s->ev[i]);
    for (int i = 0; i < 2; i++)
        if (s->ev_in[i]) cudaEventDestroy(s->ev_in[i]);
    if (s->ev_cfork) cudaEventDestroy(s->ev_cfork);
    if (s->copy_stream) cudaStreamDestroy(s->copy_stream);
    if (s->stream) cudaStreamDestroy(s->stream);
    delete s;
}

uint32_t ks_snapshot_num_nodes(const ks_snapshot* s) { return s ? s->N : 0; }
uint32_t ks_snapshot_label_words(const ks_snapshot* s) { return s ? s->W : 0; }

int ks_snapshot_set_nodes(ks_snapshot* s, uint32_t n_nodes, uint32_t label_words, const int64_t* alloc_cpu,
                          const int64_t* alloc_mem, const uint64_t* labels) {
    if (!s) return fail(KS_ERR_INVALID, "snapshot is NULL");
    if (label_words != 1 && label_words != 2 && label_words != 4 && label_words != 8)
        return fail(KS_ERR_INVALID, "label_words must be 1, 2, 4 or 8 (got %u)", label_words);
    if (n_nodes && (!alloc_cpu || !alloc_mem || !labels)) return fail(KS_ERR_INVALID, "NULL node array");
    if (n_nodes > (1u << 30)) return fail(KS_ERR_RANGE, "n_nodes too large");
    for (uint32_t n = 0; n < n_nodes; n++) {
        if (alloc_cpu[n] > KS_MAX_CPU_MILLI || alloc_cpu[n] < -KS_MAX_CPU_MILLI || alloc_mem[n] > KS_MAX_MEM_BYTES ||
            alloc_mem[n] < -KS_MAX_MEM_BYTES)
            return fail(KS_ERR_RANGE, "node %u allocatable outside +-2^36 millicores / +-2^55 bytes", n);
    }
    std::lock_guard<std::mutex> lk(s->mu);
    CU_TRY(cudaSetDevice(s->device));
    const uint32_t Npad = ((n_nodes + TILE_N - 1) / TILE_N) * TILE_N;
    s->N = n_nodes;
    s->Npad = Npad;
    s->W = label_words;
    s->derived_dirty = true;
    s->version++;
    if (Npad == 0) return KS_OK;
    std::vector<int64_t> h;
    std::vector<uint64_t> hl;
    try { // no exception crosses the ABI
        h.resize(Npad);
        hl.assign((size_t)Npad * label_words, 0);
    } catch (...) {
        return fail(KS_ERR_NOMEM, "out of host memory staging %u nodes", n_nodes);
    }
    const size_t nb = (size_t)Npad * 8;
    CU_TRY(s->alloc_cpu.ensure(nb));
    CU_TRY(s->alloc_mem.ensure(nb));
    CU_TRY(s->free_cpu.ensure(nb));
    CU_TRY(s->free_mem.ensure(nb));
    CU_TRY(s->prio.ensure(2 * nb)); // [leftover priority | least-allocated bound]
    CU_TRY(s->labels.ensure(nb * label_words));
    // allocatable: pad with 0; free: pad with INT64_MIN (never feasible)
    for (uint32_t n = 0; n < Npad; n++) h[n] = n < n_nodes ? alloc_cpu[n] : 0;
    CU_TRY(cudaMemcpyAsync(s->alloc_cpu.p, h.data(), nb, cudaMemcpyHostToDevice, s->stream));
    for (uint32_t n = n_nodes; n < Npad; n++) h[n] = INT64_MIN;
    CU_TRY(cudaMemcpyAsync(s->free_cpu.p, h.data(), nb, cudaMemcpyHostToDevice, s->stream));
    CU_TRY(cudaStreamSynchronize(s->stream));
    for (uint32_t n = 0; n < Npad; n++) h[n] = n < n_nodes ? alloc_mem[n] : 0;
    CU_TRY(cudaMemcpyAsync(s->alloc_mem.p, h.data(), nb, cudaMemcpyHostToDevice, s->stream));
    for (uint32_t n = n_nodes; n < Npad; n++) h[n] = INT64_MIN;
    CU_TRY(cudaMemcpyAsync(s->free_mem.p, h.data(), nb, cudaMemcpyHostToDevice, s->stream));
    for (uint32_t n = 0; n < n_nodes; n++)
        for (uint32_t w = 0; w < label_words; w++) hl[(size_t)w * Npad + n] = labels[(size_t)n * label_words + w];
    CU_TRY(cudaMemcpyAsync(s->labels.p, hl.data(), nb * label_words, cudaMemcpyHostToDevice, s->stream));
    CU_TRY(cudaStreamSynchronize(s->stream));
    return check_range_and_prio(s, s->stream);
}

static int reset_free_to_alloc(ks_snapshot* s) {
    // free[0..N) = alloc[0..N); the padding keeps its INT64_MIN sentinels
    CU_TRY(cudaMemcpyAsync(s->free_cpu.p, s->alloc_cpu.p, (size_t)s->N * 8, cudaMemcpyDeviceToDevice, s->stream));
    CU_TRY(cudaMemcpyAsync(s->free_mem.p, s->alloc_mem.p, (size_t)s->N * 8, cudaMemcpyDeviceToDevice, s->stream));
    return KS_OK;
}

int ks_snapshot_set_bound(ks_snapshot* s, uint64_t n_bound, const int32_t* node_idx, const int64_t* req_cpu,
                          const int64_t* req_mem) {
    if (!s) return fail(KS_ERR_INVALID, "snapshot is NULL");
    if (n_bound && (!node_idx || !req_cpu || !req_mem)) return fail(KS_ERR_INVALID, "NULL bound array");
    for (uint64_t b = 0; b < n_bound; b++) {
        if (node_idx[b] < 0 || (uint32_t)node_idx[b] >= s->N)
            return fail(KS_ERR_INVALID, "bound pod %llu: node index %d out of range", (unsigned long long)b,
                        node_idx[b]);
        if (req_cpu[b] > KS_MAX_CPU_MILLI || req_cpu[b] < -KS_MAX_CPU_MILLI || req_mem[b] > KS_MAX_MEM_BYTES ||
            req_mem[b] < -KS_MAX_MEM_BYTES)
            return fail(KS_ERR_RANGE, "bound pod %llu request out of range", (unsigned long long)b);
    }
    std::lock_guard<std::mutex> lk(s->mu);
    CU_TRY(cudaSetDevice(s->device));
    s->derived_dirty = true;
    s->version++;
    if (s->N == 0) return KS_OK;
    int rc = reset_free_to_alloc(s);
    if (rc) return rc;
    if (n_bound) {
        CU_TRY(s->st_bnode.ensure(n_bound * 4));
        CU_TRY(s->st_bcpu.ensure(n_bound * 8));
        CU_TRY(s->st_bmem.ensure(n_bound * 8));
        CU_TRY(cudaMemcpyAsync(s->st_bnode.p, node_idx, n_bound * 4, cudaMemcpyHostToDevice, s->stream));
        CU_TRY(cudaMemcpyAsync(s->st_bcpu.p, req_cpu, n_bound * 8, cudaMemcpyHostToDevice, s->stream));
        CU_TRY(cudaMemcpyAsync(s->st_bmem.p, req_mem, n_bound * 8, cudaMemcpyHostToDevice, s->stream));
        CU_TRY(launch_free_reduce(s->free_cpu.as<int64_t>(), s->free_mem.as<int64_t>(), s->st_bnode.as<int32_t>(),
                                  s->st_bcpu.as<int64_t>(), s->st_bmem.as<int64_t>(), n_bound, s->stream));
    }
    return check_range_and_prio(s, s->stream);
}

int ks_snapshot_apply_bind(ks_snapshot* s, int32_t node_idx, int64_t req_cpu, int64_t req_mem) {
    if (!s) return fail(KS_ERR_INVALID, "snapshot is NULL");
    if (node_idx < 0 || (uint32_t)node_idx >= s->N) return fail(KS_ERR_INVALID, "node index %d out of range", node_idx);
    if (req_cpu > KS_MAX_CPU_MILLI || req_cpu < -KS_MAX_CPU_MILLI || req_mem > KS_MAX_MEM_BYTES || req_mem < -KS_MAX_MEM_BYTES)
        return fail(KS_ERR_RANGE, "request out of range");
    std::lock_guard<std::mutex> lk(s->mu);
    CU_TRY(cudaSetDevice(s->device));
    s->derived_dirty = true;
    s->version++;
    CU_TRY(s->st_bnode.ensure(4));
    CU_TRY(s->st_bcpu.ensure(8));
    CU_TRY(s->st_bmem.ensure(8));
    CU_TRY(cudaMemcpyAsync(s->st_bnode.p, &node_idx, 4, cudaMemcpyHostToDevice, s->stream));
    CU_TRY(cudaMemcpyAsync(s->st_bcpu.p, &req_cpu, 8, cudaMemcpyHostToDevice, s->stream));
    CU_TRY(cudaMemcpyAsync(s->st_bmem.p, &req_mem, 8, cudaMemcpyHostToDevice, s->stream));
    CU_TRY(launch_free_reduce(s->free_cpu.as<int64_t>(), s->free_mem.as<int64_t>(), s->st_bnode.as<int32_t>(),
                              s->st_bcpu.as<int64_t>(), s->st_bmem.as<int64_t>(), 1, s->stream));
    CU_TRY(cudaStreamSynchronize(s->stream));
    return KS_OK;
}

int ks_snapshot_get_free(ks_snapshot* s, int64_t* free_cpu, int64_t* free_mem) {
    if (!s || !free_cpu || !free_mem) return fail(KS_ERR_INVALID, "NULL argument");
    std::lock_guard<std::mutex> lk(s->mu);
    CU_TRY(cudaSetDevice(s->device));
    if (s->N == 0) return KS_OK;
    CU_TRY(cudaMemcpyAsync(free_cpu, s->free_cpu.p, (size_t)s->N * 8, cudaMemcpyDeviceToHost, s->stream));
    CU_TRY(cudaMemcpyAsync(free_mem, s->free_mem.p, (size_t)s->N * 8, cudaMemcpyDeviceToHost, s->stream));
    CU_TRY(cudaStreamSynchronize(s->stream));
    return KS_OK;
}

// rebuild what depends on free[]: range check, static priorities, bit-parallel index
static int refresh_derived(ks_snapshot* s, cudaStream_t st) {
    if (!s->derived_dirty || s->N == 0) return KS_OK;
    CU_TRY(launch_node_prio(s->free_cpu.as<int64_t>(), s->free_mem.as<int64_t>(), s->prio.as<int64_t>(), s->N, s->Npad,
                            s->flag.as<int>(), st));
    cudaError_t e = bitpar_build(s->bp, node_table(s), s->prio.as<int64_t>(), st);
    if (e != cudaSuccess) return fail(KS_ERR_CUDA, "bit-parallel index build failed: %s", cudaGetErrorString(e));
    s->derived_dirty = false;
    s->version++;
    return KS_OK;
}

// host-space pods [c0, c1) into the staging buffers that stage_pods prepared
static int copy_pods_in(ks_snapshot* s, const ks_pods* pods, uint64_t c0, uint64_t c1, cudaStream_t st) {
    const uint64_t m = c1 - c0, W = s->W;
    CU_TRY(cudaMemcpyAsync(s->st_rc.as<int64_t>() + c0, pods->req_cpu + c0, m * 8, cudaMemcpyHostToDevice, st));
    CU_TRY(cudaMemcpyAsync(s->st_rm.as<int64_t>() + c0, pods->req_mem + c0, m * 8, cudaMemcpyHostToDevice, st));
    CU_TRY(cudaMemcpyAsync(s->st_sel.as<uint64_t>() + c0 * W, pods->sel + c0 * W, m * 8 * W, cudaMemcpyHostToDevice, st));
    return KS_OK;
}

static bool is_pinned_host(const void* p) {
    if (!p) return true;
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return a.type == cudaMemoryTypeHost;
}

// passing st == nullptr only prepares (allocates staging, fills *pv); the copies are enqueued by copy_pods_in
static int stage_pods(ks_snapshot* s, const ks_pods* pods, cudaStream_t st, PodView* pv) {
    const uint64_t P = pods->n;
    pv->P = (uint32_t)P;
    if (pods->mem_space == KS_MEM_DEVICE) {
        pv->req_cpu = pods->req_cpu;
        pv->req_mem = pods->req_mem;
        pv->sel = pods->sel;
        return KS_OK;
    }
    CU_TRY(s->st_rc.ensure(P * 8));
    CU_TRY(s->st_rm.ensure(P * 8));
    CU_TRY(s->st_sel.ensure(P * 8 * s->W));
    pv->req_cpu = s->st_rc.as<int64_t>();
    pv->req_mem = s->st_rm.as<int64_t>();
    pv->sel = s->st_sel.as<uint64_t>();
    if (st == nullptr) return KS_OK; // prepare only: the caller enqueues the copies itself (copy_pods_in)
    return copy_pods_in(s, pods, 0, P, st);
}

static int check_pods(const ks_snapshot* s, const ks_pods* pods) {
    if (!s) return fail(KS_ERR_INVALID, "snapshot is NULL");
    if (!pods) return fail(KS_ERR_INVALID, "pods is NULL");
    if (pods->n > 0xfffffff0ull) return fail(KS_ERR_RANGE, "too many pods in one call");
    if (pods->n && (!pods->req_cpu || !pods->req_mem || !pods->sel)) return fail(KS_ERR_INVALID, "NULL pod array");
    if (pods->mem_space != KS_MEM_HOST && pods->mem_space != KS_MEM_DEVICE)
        return fail(KS_ERR_INVALID, "bad pods.mem_space");
    return KS_OK;
}

int ks_check_cells(ks_snapshot* s, const ks_pods* pods, uint8_t* out_codes) {
    int rc = check_pods(s, pods);
    if (rc) return rc;
    if (!out_codes) return fail(KS_ERR_INVALID, "out_codes is NULL");
    const uint64_t cells = pods->n * (uint64_t)s->N;
    if (cells == 0) return KS_OK;
    if (cells > (1ull << 31)) return fail(KS_ERR_RANGE, "ks_check_cells is for <= 2^31 cells");
    std::lock_guard<std::mutex> lk(s->mu);
    CU_TRY(cudaSetDevice(s->device));
    PodView pv;
    rc = stage_pods(s, pods, s->stream, &pv);
    if (rc) return rc;
    CU_TRY(s->st_codes.ensure(cells));
    CU_TRY(launch_check_cells(node_table(s), pv, s->st_codes.as<uint8_t>(), 0, s->N, s->stream));
    CU_TRY(cudaMemcpyAsync(out_codes, s->st_codes.p, cells, cudaMemcpyDeviceToHost, s->stream));
    CU_TRY(cudaStreamSynchronize(s->stream));
    return KS_OK;
}

int ks_check_cell(ks_snapshot* s, int64_t req_cpu, int64_t req_mem, const uint64_t* sel, uint32_t node_idx) {
    if (!s || !sel) return fail(KS_ERR_INVALID, "NULL argument");
    if (node_idx >= s->N) return fail(KS_ERR_INVALID, "node index %u out of range", node_idx);
    std::lock_guard<std::mutex> lk(s->mu);
    CU_TRY(cudaSetDevice(s->device));
    ks_pods pods;
    pods.n = 1;
    pods.req_cpu = &req_cpu;
    pods.req_mem = &req_mem;
    pods.sel = sel;
    pods.mem_space = KS_MEM_HOST;
    PodView pv;
    int rc = stage_pods(s, &pods, s->stream, &pv);
    if (rc) return rc;
    CU_TRY(s->st_codes.ensure(16));
    CU_TRY(launch_check_cells(node_table(s), pv, s->st_codes.as<uint8_t>(), node_idx, 1, s->stream));
    uint8_t code = 0xff;
    CU_TRY(cudaMemcpyAsync(&code, s->st_codes.p, 1, cudaMemcpyDeviceToHost, s->stream));
    CU_TRY(cudaStreamSynchronize(s->stream));
    return (int)code;
}

static int check_select_args(const ks_snapshot* s, const ks_pods* pods, int policy, uint32_t flags, const ks_bindings* out) {
    int rc = check_pods(s, pods);
    if (rc) return rc;
    if (!out) return fail(KS_ERR_INVALID, "out is NULL");
    if (policy != KS_SCORE_LEFTOVER && policy != KS_SCORE_LEAST_ALLOCATED) return fail(KS_ERR_INVALID, "bad policy");
    if ((flags & KS_SELECT_FORCE_BITPAR) && (flags & KS_SELECT_FORCE_DIRECT)) return fail(KS_ERR_INVALID, "bad flags");
    if (out->mask) {
        if (out->mask_row_bytes % 32 != 0 || out->mask_row_bytes < ks_mask_row_bytes(s->N))
            return fail(KS_ERR_INVALID, "mask_row_bytes must be a multiple of 32 and >= %llu",
                        (unsigned long long)ks_mask_row_bytes(s->N));
        if (out->mask_space == KS_MEM_DEVICE && ((uintptr_t)out->mask & 31u) != 0)
            return fail(KS_ERR_INVALID, "a device-space mask must be 32-byte aligned");
    }
    const ks_exchange* xc = out->exchange;
    if (xc) {
        if (out->mem_space != KS_MEM_DEVICE || !out->node_idx || !out->score)
            return fail(KS_ERR_INVALID, "exchange needs device-space node_idx and score outputs");
        if (xc->world < 2 || xc->world > KS_MAX_PEERS + 1 || xc->rank >= xc->world || xc->n_peers != xc->world - 1)
            return fail(KS_ERR_INVALID, "bad exchange world/rank/n_peers");
        if (!xc->local_flags || !xc->local_state) return fail(KS_ERR_INVALID, "exchange: NULL local_flags / local_state");
        for (uint32_t k = 0; k < xc->n_peers; k++)
            if (!xc->peer_node_idx[k] || !xc->peer_score[k] || !xc->peer_flag[k])
                return fail(KS_ERR_INVALID, "exchange: NULL peer pointer %u", k);
    }
    return KS_OK;
}

static PeerOut peer_out(const ks_exchange* xc) {
    PeerOut po;
    if (!xc) return po;
    po.n = xc->n_peers;
    po.world = xc->world;
    po.rank = xc->rank;
    for (uint32_t k = 0; k < xc->n_peers; k++) {
        po.idx[k] = xc->peer_node_idx[k];
        po.score[k] = xc->peer_score[k];
        po.flag[k] = xc->peer_flag[k];
    }
    po.local_flags = xc->local_flags;
    po.state = xc->local_state;
    return po;
}

struct SelectPlan {
    SelectPath path;
    SelectLaunch L;                        // the whole call; host-space outputs point to their device staging
    PartialView part;                      // direct path: partial results per node chunk
    uint32_t node_chunks, tiles_per_chunk; // direct path: split of the node dimension across CTAs
    uint32_t pod_chunks;                   // 2 = the host-space pipeline, else 1
};

// Picks the path and the pod chunking and makes every allocation of the call: the launch sequence that follows may be
// stream-captured, and nothing may allocate inside a capture.
static int plan_select(ks_snapshot* s, const ks_pods* pods, int policy, uint32_t flags, const ks_bindings* out,
                       const PeerOut& po, cudaStream_t st, SelectPlan* pl) {
    const uint64_t P = pods->n;
    // the per-cell kernel needs no derived state; the bit-parallel index is (re)built lazily
    const bool may_bitpar = (flags & KS_SELECT_FORCE_BITPAR) ||
                            (!(flags & KS_SELECT_FORCE_DIRECT) && P * s->N >= (1ull << 24));
    if (may_bitpar) {
        const int rc = refresh_derived(s, st);
        if (rc) return rc;
    }
    SelectLaunch& L = pl->L;
    L.nt = node_table(s);
    L.pv.P = (uint32_t)P;
    L.policy = policy;
    L.stream = st;
    L.po = po;
    OutView& ov = L.ov;
    ov.node_idx = out->node_idx;
    ov.score = out->score;
    ov.cnt = out->feasible_cnt;
    ov.mask = reinterpret_cast<uint32_t*>(out->mask);
    ov.mask_row_words = out->mask_row_bytes / 4;
    ov.mask_valid_words = (uint32_t)(ks_mask_row_bytes(s->N) / 4);
    const bool out_host = out->mem_space == KS_MEM_HOST;
    const bool mask_host = out->mask && out->mask_space == KS_MEM_HOST;
    if (out_host) {
        if (out->node_idx) {
            CU_TRY(s->st_idx.ensure(P * 4));
            ov.node_idx = s->st_idx.as<int32_t>();
        }
        if (out->score) {
            CU_TRY(s->st_score.ensure(P * 8));
            ov.score = s->st_score.as<int64_t>();
        }
        if (out->feasible_cnt) {
            CU_TRY(s->st_cnt.ensure(P * 4));
            ov.cnt = s->st_cnt.as<uint32_t>();
        }
    }
    if (mask_host) {
        CU_TRY(s->st_mask.ensure(P * out->mask_row_bytes));
        ov.mask = s->st_mask.as<uint32_t>();
    }
    pl->pod_chunks = 1;
    if (s->N == 0) {
        pl->path = PATH_EMPTY;
        s->last_path = "empty";
        return KS_OK;
    }
    int rc = stage_pods(s, pods, nullptr, &L.pv);
    if (rc) return rc;
    bool use_bitpar = false;
    if (flags & KS_SELECT_FORCE_BITPAR) use_bitpar = true;
    else if (!(flags & KS_SELECT_FORCE_DIRECT))
        use_bitpar = may_bitpar && bitpar_profitable(s->bp, L.pv.P);
    if (use_bitpar) {
        cudaError_t e = bitpar_prepare(s->bp, L.pv.P);
        if (e != cudaSuccess) return fail(KS_ERR_CUDA, "bit-parallel prepare failed: %s", cudaGetErrorString(e));
    } else {
        const uint32_t n_tiles = s->Npad / TILE_N;
        const uint32_t pod_ctas = (L.pv.P + direct_pods_per_cta(s->W) - 1) / direct_pods_per_cta(s->W);
        const uint32_t want_ctas = 2u * (uint32_t)s->sms; // at least two CTAs per SM
        uint32_t n_chunks = 1;
        if (pod_ctas < want_ctas) n_chunks = std::min<uint32_t>(n_tiles, (want_ctas + pod_ctas - 1) / pod_ctas);
        pl->tiles_per_chunk = (n_tiles + n_chunks - 1) / n_chunks;
        pl->node_chunks = (n_tiles + pl->tiles_per_chunk - 1) / pl->tiles_per_chunk;
        if (pl->node_chunks > 1) {
            CU_TRY(s->part_key.ensure((size_t)pl->node_chunks * P * 8));
            CU_TRY(s->part_idx.ensure((size_t)pl->node_chunks * P * 4));
            CU_TRY(s->part_cnt.ensure((size_t)pl->node_chunks * P * 4));
            pl->part.key = s->part_key.as<int64_t>();
            pl->part.idx = s->part_idx.as<int32_t>();
            pl->part.cnt = s->part_cnt.as<uint32_t>();
        }
        cudaError_t e = prepare_select_direct(s->W);
        if (e != cudaSuccess) return fail(KS_ERR_CUDA, "direct prepare failed: %s", cudaGetErrorString(e));
    }
    pl->path = use_bitpar ? PATH_BITPAR : PATH_DIRECT;
    s->last_path = use_bitpar ? "bitpar" : "direct";
    // Host-space batches on the bit-parallel path are pipelined in two pod chunks: the second chunk is copied in on
    // copy_stream while the first computes, and the bindings of a chunk travel back under the next chunk's mask kernel.
    // (Each chunk is an independent select over its pod range; scratch is reused because a chunk starts only after the
    // previous chunk's auxiliary-stream work has joined.)
    if (use_bitpar && pods->mem_space == KS_MEM_HOST && out_host && !mask_host && !(flags & KS_SELECT_TIMING) &&
        P >= 262144) // below that the per-chunk launch overhead outweighs the overlap (measured at 100k pods)
        pl->pod_chunks = 2;
    return KS_OK;
}

// One pod chunk of the planned path.  Clears what it served of Lc.host_node_idx / host_score / ready_event.
static int launch_chunk(ks_snapshot* s, const SelectPlan& pl, SelectLaunch& Lc, bool timing) {
    const cudaStream_t st = Lc.stream;
    const uint64_t m = Lc.pv.P;
    cudaError_t e = cudaSuccess;
    switch (pl.path) {
        case PATH_EMPTY: // every pod gets None (src/main.rs:56,70)
            if (Lc.ov.node_idx) CU_TRY(cudaMemsetAsync(Lc.ov.node_idx, 0xff, m * 4, st));
            if (Lc.ov.score) CU_TRY(cudaMemsetAsync(Lc.ov.score, 0, m * 8, st));
            if (Lc.ov.cnt) CU_TRY(cudaMemsetAsync(Lc.ov.cnt, 0, m * 4, st));
            CU_TRY(launch_exchange_push(Lc.po, Lc.ov.node_idx, Lc.ov.score, (uint32_t)m, st));
            break;
        case PATH_DIRECT:
            if (timing) CU_TRY(cudaEventRecord(s->ev[1], st));
            e = launch_select_direct(Lc, pl.part, pl.node_chunks, pl.tiles_per_chunk);
            if (e != cudaSuccess) return fail(KS_ERR_CUDA, "direct select failed: %s", cudaGetErrorString(e));
            if (timing) CU_TRY(cudaEventRecord(s->ev[2], st));
            CU_TRY(launch_exchange_push(Lc.po, Lc.ov.node_idx, Lc.ov.score, (uint32_t)m, st));
            break;
        case PATH_BITPAR: // the argmax kernels send the bindings to the peers themselves
            e = bitpar_select(s->bp, Lc, timing ? s->ev[1] : nullptr, timing ? s->ev[2] : nullptr);
            if (e != cudaSuccess) return fail(KS_ERR_CUDA, "bit-parallel select failed: %s", cudaGetErrorString(e));
            break;
    }
    return KS_OK;
}

// The launch sequence of a planned ks_select: per pod chunk, wait for its input copy, launch it, copy back the host
// outputs the launcher has not served; then the per-call tail.  Allocates nothing.
static int enqueue_select(ks_snapshot* s, const ks_pods* pods, const ks_bindings* out, const SelectPlan& pl, bool timing) {
    const SelectLaunch& L = pl.L;
    const cudaStream_t st = L.stream;
    const uint64_t P = L.pv.P, W = s->W;
    const uint32_t n = pl.pod_chunks;
    const bool out_host = out->mem_space == KS_MEM_HOST;
    if (pl.path != PATH_EMPTY && pods->mem_space == KS_MEM_HOST) {
        const cudaStream_t cs = n > 1 ? s->copy_stream : st;
        if (n > 1) {
            CU_TRY(cudaEventRecord(s->ev_cfork, st));
            CU_TRY(cudaStreamWaitEvent(cs, s->ev_cfork, 0));
        }
        for (uint32_t c = 0; c < n; c++) {
            const int rc = copy_pods_in(s, pods, P * c / n, P * (c + 1) / n, cs);
            if (rc) return rc;
            if (n > 1) CU_TRY(cudaEventRecord(s->ev_in[c], cs));
        }
    }
    cudaEvent_t ready = out_host ? nullptr : (cudaEvent_t)out->bindings_ready_event;
    for (uint32_t c = 0; c < n; c++) {
        const uint64_t c0 = P * c / n, m = P * (c + 1) / n - c0;
        if (n > 1) CU_TRY(cudaStreamWaitEvent(st, s->ev_in[c], 0));
        SelectLaunch Lc = L;
        Lc.pv.req_cpu += c0;
        Lc.pv.req_mem += c0;
        Lc.pv.sel += c0 * W;
        Lc.pv.P = (uint32_t)m;
        if (Lc.ov.node_idx) Lc.ov.node_idx += c0;
        if (Lc.ov.score) Lc.ov.score += c0;
        if (Lc.ov.cnt) Lc.ov.cnt += c0;
        if (Lc.ov.mask) Lc.ov.mask += c0 * Lc.ov.mask_row_words;
        Lc.host_node_idx = out_host && out->node_idx ? out->node_idx + c0 : nullptr;
        Lc.host_score = out_host && out->score ? out->score + c0 : nullptr;
        Lc.ready_event = ready;
        const int rc = launch_chunk(s, pl, Lc, timing);
        if (rc) return rc;
        ready = Lc.ready_event;
        if (Lc.host_node_idx) CU_TRY(cudaMemcpyAsync(Lc.host_node_idx, Lc.ov.node_idx, m * 4, cudaMemcpyDeviceToHost, st));
        if (Lc.host_score) CU_TRY(cudaMemcpyAsync(Lc.host_score, Lc.ov.score, m * 8, cudaMemcpyDeviceToHost, st));
        if (out_host && out->feasible_cnt)
            CU_TRY(cudaMemcpyAsync(out->feasible_cnt + c0, Lc.ov.cnt, m * 4, cudaMemcpyDeviceToHost, st));
    }
    // The per-call tail runs once, after the last chunk.  Two chunks need host-space outputs and no host-space mask, while
    // an exchange and a ready event need device-space outputs: with two chunks the tail has nothing to do.
    // With an exchange, the call's stream work ends when every other rank's bindings have arrived here.
    CU_TRY(launch_exchange_wait(L.po, s->xflag.as<int>(), st));
    if (out->mask && out->mask_space == KS_MEM_HOST && pl.path != PATH_EMPTY) // the empty store writes no mask
        CU_TRY(cudaMemcpyAsync(out->mask, L.ov.mask, P * out->mask_row_bytes, cudaMemcpyDeviceToHost, st));
    if (ready) CU_TRY(record_ready_event(ready, st)); // not served by the launcher: the bindings are final here
    return KS_OK;
}

static SelectKey select_key(const ks_snapshot* s, const ks_pods* pods, int policy, uint32_t flags, const ks_bindings* out,
                            cudaStream_t st, SelectPath path) {
    SelectKey k{};
    k.P = pods->n;
    k.req_cpu = pods->req_cpu;
    k.req_mem = pods->req_mem;
    k.sel = pods->sel;
    k.node_idx = out->node_idx;
    k.score = out->score;
    k.feasible_cnt = out->feasible_cnt;
    k.mask = out->mask;
    k.mask_row_bytes = out->mask_row_bytes;
    k.policy = policy;
    k.pods_space = pods->mem_space;
    k.out_space = out->mem_space;
    k.mask_space = out->mask_space;
    k.flags = flags;
    k.path = path;
    k.stream = st;
    k.ready_event = out->bindings_ready_event;
    k.version = s->version;
    k.devbuf_epoch = g_devbuf_epoch.load();
    k.bitpar_epoch = s->bp.epoch;
    if (const ks_exchange* xc = out->exchange) {
        k.world = xc->world;
        k.rank = xc->rank;
        k.n_peers = xc->n_peers;
        for (uint32_t i = 0; i < xc->n_peers; i++) {
            k.peer_node_idx[i] = xc->peer_node_idx[i];
            k.peer_score[i] = xc->peer_score[i];
            k.peer_flag[i] = xc->peer_flag[i];
        }
        k.local_flags = xc->local_flags;
        k.local_state = xc->local_state;
    }
    return k;
}

// a captured copy from pageable host memory is not allowed: a call with host-space buffers is replayed only if they are pinned
static bool host_buffers_pinned(const ks_pods* pods, const ks_bindings* out) {
    if (pods->mem_space == KS_MEM_HOST &&
        !(is_pinned_host(pods->req_cpu) && is_pinned_host(pods->req_mem) && is_pinned_host(pods->sel)))
        return false;
    if (out->mem_space == KS_MEM_HOST &&
        !(is_pinned_host(out->node_idx) && is_pinned_host(out->score) && is_pinned_host(out->feasible_cnt)))
        return false;
    return !(out->mask && out->mask_space == KS_MEM_HOST) || is_pinned_host(out->mask);
}

int ks_select(ks_snapshot* s, const ks_pods* pods, int policy, uint32_t flags, ks_bindings* out, void* cuda_stream) {
    int rc = check_select_args(s, pods, policy, flags, out);
    if (rc) return rc;
    const uint64_t P = pods->n;
    if (P == 0 && !out->exchange) return KS_OK;
    std::lock_guard<std::mutex> lk(s->mu);
    CU_TRY(cudaSetDevice(s->device));
    cudaStream_t st = cuda_stream ? (cudaStream_t)cuda_stream : s->stream;
    const bool timing = (flags & KS_SELECT_TIMING) != 0;
    const PeerOut po = peer_out(out->exchange);
    if (P == 0) { // an empty shard still takes part in the exchange: publish the sequence number, wait for the others
        CU_TRY(launch_exchange_push(po, nullptr, nullptr, 0, st));
        CU_TRY(launch_exchange_wait(po, s->xflag.as<int>(), st));
        return KS_OK;
    }
    s->timing_valid = false;
    if (timing) CU_TRY(cudaEventRecord(s->ev[0], st));
    SelectPlan pl{};
    rc = plan_select(s, pods, policy, flags, out, po, st, &pl);
    if (rc) return rc;
    auto enqueue = [&] { return enqueue_select(s, pods, out, pl, timing); };
    // The kernel paths replay a repeated call from the cached CUDA graph; the pinned check only runs on a key miss.
    const SelectKey key = select_key(s, pods, policy, flags, out, st, pl.path);
    if (pl.path != PATH_EMPTY && !timing && !(flags & KS_SELECT_NO_GRAPH) &&
        (s->graph.hit(key) || host_buffers_pinned(pods, out)))
        rc = s->graph.run(key, st, enqueue);
    else
        rc = enqueue();
    if (rc) return rc;
    if (timing) {
        CU_TRY(cudaEventRecord(s->ev[3], st));
        s->timing_valid = s->N != 0;
    }
    const bool mask_host = out->mask && out->mask_space == KS_MEM_HOST;
    if (out->mem_space == KS_MEM_HOST || mask_host || pods->mem_space == KS_MEM_HOST || timing)
        CU_TRY(cudaStreamSynchronize(st));
    return KS_OK;
}

int ks_last_timings(ks_snapshot* s, float ms[3]) {
    if (!s || !ms) return fail(KS_ERR_INVALID, "NULL argument");
    if (!s->timing_valid) return fail(KS_ERR_INVALID, "no KS_SELECT_TIMING call recorded");
    CU_TRY(cudaSetDevice(s->device));
    CU_TRY(cudaEventSynchronize(s->ev[3]));
    CU_TRY(cudaEventElapsedTime(&ms[0], s->ev[1], s->ev[2]));
    CU_TRY(cudaEventElapsedTime(&ms[1], s->ev[2], s->ev[3]));
    CU_TRY(cudaEventElapsedTime(&ms[2], s->ev[0], s->ev[3]));
    return KS_OK;
}

const char* ks_last_path(const ks_snapshot* s) { return s ? s->last_path : "none"; }

int ks_last_trace(ks_snapshot* s, uint64_t out_ns[16]) {
    if (!s || !out_ns) return fail(KS_ERR_INVALID, "NULL argument");
    static_assert(BP_TRACE_WORDS == 16, "ks_last_trace layout");
    CU_TRY(cudaSetDevice(s->device));
    unsigned long long tmp[BP_TRACE_WORDS];
    const cudaError_t e = bitpar_read_trace(s->bp, tmp);
    if (e == cudaErrorNotSupported) return fail(KS_ERR_INVALID, "no trace: run the process with KS_TRACE=1");
    if (e != cudaSuccess) return fail(KS_ERR_CUDA, "trace read failed: %s", cudaGetErrorString(e));
    for (int k = 0; k < BP_TRACE_WORDS; k++) out_ns[k] = tmp[k];
    return KS_OK;
}

int ks_exchange_check(ks_snapshot* s) {
    if (!s) return fail(KS_ERR_INVALID, "snapshot is NULL");
    std::lock_guard<std::mutex> lk(s->mu);
    CU_TRY(cudaSetDevice(s->device));
    CU_TRY(cudaDeviceSynchronize());
    int flag = 0;
    CU_TRY(cudaMemcpy(&flag, s->xflag.p, sizeof(int), cudaMemcpyDeviceToHost));
    if (flag) {
        CU_TRY(cudaMemset(s->xflag.p, 0, sizeof(int)));
        return fail(KS_ERR_CUDA, "exchange: a peer's bindings did not arrive within the timeout");
    }
    return KS_OK;
}

int ks_ipc_alloc(int device, uint64_t bytes, void** out_ptr, uint8_t out_handle[64]) {
    if (!out_ptr || !out_handle || bytes == 0) return fail(KS_ERR_INVALID, "bad ks_ipc_alloc argument");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
    CU_TRY(cudaSetDevice(device));
    void* p = nullptr;
    CU_TRY(cudaMalloc(&p, bytes));
    cudaError_t e = cudaMemset(p, 0, bytes);
    cudaIpcMemHandle_t h;
    if (e == cudaSuccess) e = cudaIpcGetMemHandle(&h, p);
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (e != cudaSuccess) {
        cudaFree(p);
        return fail(KS_ERR_CUDA, "ks_ipc_alloc failed: %s", cudaGetErrorString(e));
    }
    memcpy(out_handle, &h, 64);
    *out_ptr = p;
    return KS_OK;
}

int ks_ipc_open(int device, const uint8_t handle[64], void** out_ptr) {
    if (!out_ptr || !handle) return fail(KS_ERR_INVALID, "bad ks_ipc_open argument");
    CU_TRY(cudaSetDevice(device));
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, 64);
    CU_TRY(cudaIpcOpenMemHandle(out_ptr, h, cudaIpcMemLazyEnablePeerAccess));
    return KS_OK;
}

int ks_ipc_close(int device, void* ptr) {
    if (!ptr) return KS_OK;
    CU_TRY(cudaSetDevice(device));
    CU_TRY(cudaIpcCloseMemHandle(ptr));
    return KS_OK;
}

int ks_measure_write_bandwidth(int device, void* dev_buf, uint64_t bytes, int iters, double* out_gbs) {
    if (!dev_buf || !out_gbs || bytes < (1u << 20) || ((uintptr_t)dev_buf & 31u)) return fail(KS_ERR_INVALID, "bad argument");
    CU_TRY(cudaSetDevice(device));
    int sms = 0;
    CU_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
    cudaEvent_t e0, e1;
    CU_TRY(cudaEventCreate(&e0));
    CU_TRY(cudaEventCreate(&e1));
    float best = 1e30f;
    for (int it = 0; it < std::max(2, iters); it++) { // first pass untimed
        CU_TRY(cudaEventRecord(e0, nullptr));
        CU_TRY(launch_fill256(dev_buf, bytes, 0x5a5a0000u + (uint32_t)it, sms, nullptr));
        CU_TRY(cudaEventRecord(e1, nullptr));
        CU_TRY(cudaEventSynchronize(e1));
        float ms = 0;
        CU_TRY(cudaEventElapsedTime(&ms, e0, e1));
        if (it > 0) best = std::min(best, ms);
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    *out_gbs = (double)(bytes / 32 * 32) / (best * 1e-3) / 1e9;
    return KS_OK;
}

int ks_device_read(int device, const void* dev_ptr, void* host_ptr, uint64_t bytes) {
    if (!dev_ptr || !host_ptr) return fail(KS_ERR_INVALID, "NULL argument");
    CU_TRY(cudaSetDevice(device));
    CU_TRY(cudaDeviceSynchronize());
    CU_TRY(cudaMemcpy(host_ptr, dev_ptr, bytes, cudaMemcpyDeviceToHost));
    return KS_OK;
}

int ks_ipc_free(int device, void* ptr) {
    if (!ptr) return KS_OK;
    CU_TRY(cudaSetDevice(device));
    CU_TRY(cudaFree(ptr));
    return KS_OK;
}

int ks_snapshot_commit_claims(ks_snapshot* s, uint64_t n, const int32_t* claim_node, const int64_t* req_cpu,
                              const int64_t* req_mem, uint8_t* out_accepted) {
    if (!s) return fail(KS_ERR_INVALID, "snapshot is NULL");
    if (n && (!claim_node || !req_cpu || !req_mem || !out_accepted)) return fail(KS_ERR_INVALID, "NULL claim array");
    if (n == 0) return KS_OK;
    std::lock_guard<std::mutex> lk(s->mu);
    CU_TRY(cudaSetDevice(s->device));
    s->derived_dirty = true;
    s->version++;
    const uint32_t chunk = stream_max_claims();
    CU_TRY(s->st_bnode.ensure(n * 4));
    CU_TRY(s->st_bcpu.ensure(n * 8));
    CU_TRY(s->st_bmem.ensure(n * 8));
    CU_TRY(s->st_codes.ensure(n));
    CU_TRY(cudaMemcpyAsync(s->st_bnode.p, claim_node, n * 4, cudaMemcpyHostToDevice, s->stream));
    CU_TRY(cudaMemcpyAsync(s->st_bcpu.p, req_cpu, n * 8, cudaMemcpyHostToDevice, s->stream));
    CU_TRY(cudaMemcpyAsync(s->st_bmem.p, req_mem, n * 8, cudaMemcpyHostToDevice, s->stream));
    // chunks run in arrival order on one stream: per-node arrival order is preserved across chunks
    for (uint64_t off = 0; off < n; off += chunk) {
        const uint32_t m = (uint32_t)std::min<uint64_t>(chunk, n - off);
        CU_TRY(launch_stream_resolve(s->free_cpu.as<int64_t>(), s->free_mem.as<int64_t>(), s->st_bnode.as<int32_t>() + off,
                                     s->st_bcpu.as<int64_t>() + off, s->st_bmem.as<int64_t>() + off, m, s->N,
                                     s->st_codes.as<uint8_t>() + off, s->stream));
    }
    CU_TRY(cudaMemcpyAsync(out_accepted, s->st_codes.p, n, cudaMemcpyDeviceToHost, s->stream));
    CU_TRY(cudaStreamSynchronize(s->stream));
    return KS_OK;
}

int ks_select_sampling(ks_snapshot* s, const ks_pods* pods, uint32_t attempts, uint64_t seed, uint64_t first_pod_index,
                       int32_t* out_node_idx, uint32_t* out_attempts, int32_t* out_draw_node, uint8_t* out_draw_code) {
    int rc = check_pods(s, pods);
    if (rc) return rc;
    const uint64_t P = pods->n;
    if (P && !out_node_idx) return fail(KS_ERR_INVALID, "out_node_idx is NULL");
    if (attempts > 64) return fail(KS_ERR_RANGE, "attempts must be <= 64 (the reference uses %u)", KS_REFERENCE_ATTEMPTS);
    if (P == 0) return KS_OK;
    const uint64_t draws = P * (uint64_t)attempts;
    std::lock_guard<std::mutex> lk(s->mu);
    if (s->N == 0 || attempts == 0) { // choose() on an empty store is None for every attempt (main.rs:56,60)
        for (uint64_t i = 0; i < P; i++) out_node_idx[i] = -1;
        if (out_attempts) memset(out_attempts, 0, P * 4);
        if (out_draw_node) memset(out_draw_node, 0xff, draws * 4);
        if (out_draw_code) memset(out_draw_code, 0xff, draws);
        return KS_OK;
    }
    CU_TRY(cudaSetDevice(s->device));
    PodView pv;
    rc = stage_pods(s, pods, s->stream, &pv);
    if (rc) return rc;
    // one scratch buffer: node_idx[P] | attempts[P] | draw_node[P*attempts] | draw_code[P*attempts]
    const size_t off_att = P * 4, off_dn = off_att + P * 4, off_dc = off_dn + draws * 4;
    CU_TRY(s->st_samp.ensure(off_dc + draws));
    uint8_t* base = s->st_samp.as<uint8_t>();
    CU_TRY(launch_select_sampling(node_table(s), pv, attempts, seed, first_pod_index, reinterpret_cast<int32_t*>(base),
                                  reinterpret_cast<uint32_t*>(base + off_att),
                                  out_draw_node ? reinterpret_cast<int32_t*>(base + off_dn) : nullptr,
                                  out_draw_code ? base + off_dc : nullptr, s->stream));
    CU_TRY(cudaMemcpyAsync(out_node_idx, base, P * 4, cudaMemcpyDeviceToHost, s->stream));
    if (out_attempts) CU_TRY(cudaMemcpyAsync(out_attempts, base + off_att, P * 4, cudaMemcpyDeviceToHost, s->stream));
    if (out_draw_node) CU_TRY(cudaMemcpyAsync(out_draw_node, base + off_dn, draws * 4, cudaMemcpyDeviceToHost, s->stream));
    if (out_draw_code) CU_TRY(cudaMemcpyAsync(out_draw_code, base + off_dc, draws, cudaMemcpyDeviceToHost, s->stream));
    CU_TRY(cudaStreamSynchronize(s->stream));
    return KS_OK;
}

int ks_stream_bind(ks_snapshot* s, const ks_pods* pods, int policy, int32_t* out_node_idx, int64_t* out_score,
                   uint32_t* out_rounds) {
    int rc = check_pods(s, pods);
    if (rc) return rc;
    if (pods->mem_space != KS_MEM_HOST) return fail(KS_ERR_INVALID, "ks_stream_bind takes host-space pods");
    if (pods->n && !out_node_idx) return fail(KS_ERR_INVALID, "out_node_idx is NULL");
    const uint64_t n = pods->n;
    const uint32_t W = s->W;
    if (policy != KS_SCORE_LEFTOVER && policy != KS_SCORE_LEAST_ALLOCATED) return fail(KS_ERR_INVALID, "bad policy");
    if (n > 0 && n <= STREAM_BATCH_MAX && s->N > 0 && s->coop) {
        // device-side loop: one H2D, ONE cooperative launch that runs every round, one D2H
        std::lock_guard<std::mutex> lk(s->mu);
        CU_TRY(cudaSetDevice(s->device));
        // one pinned staging block: inputs [rc | rm | sel] and results [score | idx | ctl] are contiguous, so the whole
        // micro-batch costs ONE H2D copy, ONE cooperative launch and ONE D2H copy
        const size_t in_bytes = n * (16 + 8 * (size_t)W), o_score = 0, o_idx = n * 8, o_ctl = o_idx + ((n * 4 + 7) & ~(size_t)7),
                     out_bytes = o_ctl + 8;
        const size_t h_cap = (size_t)STREAM_BATCH_MAX * (16 + 8 * KS_MAX_LABEL_WORDS) + (size_t)STREAM_BATCH_MAX * 12 + 64;
        if (!s->h_stream) CU_TRY(cudaHostAlloc(&s->h_stream, h_cap, cudaHostAllocDefault));
        uint8_t* h_in = static_cast<uint8_t*>(s->h_stream);
        uint8_t* h_out = h_in + (size_t)STREAM_BATCH_MAX * (16 + 8 * KS_MAX_LABEL_WORDS);
        memcpy(h_in, pods->req_cpu, n * 8);
        memcpy(h_in + n * 8, pods->req_mem, n * 8);
        memcpy(h_in + n * 16, pods->sel, n * 8 * W);
        const uint32_t grid = std::max(1u, std::min<uint32_t>((uint32_t)s->sms, (s->N + 127u) / 128u));
        CU_TRY(s->st_rc.ensure((size_t)STREAM_BATCH_MAX * (16 + 8 * KS_MAX_LABEL_WORDS))); // device copy of the input block
        CU_TRY(s->st_score.ensure((size_t)STREAM_BATCH_MAX * 12 + 64));                      // device copy of the result block
        CU_TRY(s->sb_pkey.ensure((size_t)STREAM_BATCH_MAX * s->sms * 8));
        CU_TRY(s->sb_pidx.ensure((size_t)STREAM_BATCH_MAX * s->sms * 4));
        CU_TRY(s->sb_pend.ensure(2 * STREAM_BATCH_MAX * 4));
        cudaStream_t st = s->stream;
        uint8_t* d_in = s->st_rc.as<uint8_t>();
        uint8_t* d_out = s->st_score.as<uint8_t>();
        CU_TRY(cudaMemcpyAsync(d_in, h_in, in_bytes, cudaMemcpyHostToDevice, st));
        StreamBatchArgs a;
        a.N = s->N;
        a.Npad = s->Npad;
        a.alloc_cpu = s->alloc_cpu.as<int64_t>();
        a.alloc_mem = s->alloc_mem.as<int64_t>();
        a.labels = s->labels.as<uint64_t>();
        a.free_cpu = s->free_cpu.as<int64_t>();
        a.free_mem = s->free_mem.as<int64_t>();
        a.policy = policy;
        a.m = (uint32_t)n;
        a.req_cpu = reinterpret_cast<const int64_t*>(d_in);
        a.req_mem = reinterpret_cast<const int64_t*>(d_in + n * 8);
        a.sel = reinterpret_cast<const uint64_t*>(d_in + n * 16);
        a.pkey = s->sb_pkey.as<int64_t>();
        a.pidx = s->sb_pidx.as<int32_t>();
        a.pend = s->sb_pend.as<uint32_t>();
        a.ctl = reinterpret_cast<uint32_t*>(d_out + o_ctl);
        a.out_idx = reinterpret_cast<int32_t*>(d_out + o_idx);
        a.out_score = reinterpret_cast<int64_t*>(d_out + o_score);
        a.max_rounds = (uint32_t)n + 1;
        a.grid = grid;
        s->derived_dirty = true; // free[] changes: the bit-parallel index is stale
        s->version++;
        cudaError_t e = launch_stream_batch(a, W, st);
        if (e != cudaSuccess) return fail(KS_ERR_CUDA, "k_stream_batch launch failed: %s", cudaGetErrorString(e));
        CU_TRY(cudaMemcpyAsync(h_out, d_out, out_bytes, cudaMemcpyDeviceToHost, st));
        CU_TRY(cudaStreamSynchronize(st));
        memcpy(out_node_idx, h_out + o_idx, n * 4);
        if (out_score) memcpy(out_score, h_out + o_score, n * 8);
        if (out_rounds) *out_rounds = reinterpret_cast<const uint32_t*>(h_out + o_ctl)[1];
        s->last_path = "stream_batch";
        return KS_OK;
    }
    try { // host-driven loop (large batches, no cooperative launch): its vectors must not throw across the ABI
        std::vector<uint64_t> pending(n);
        for (uint64_t i = 0; i < n; i++) {
            pending[i] = i;
            out_node_idx[i] = -1;
            if (out_score) out_score[i] = 0;
        }
        std::vector<int64_t> rc_, rm_, score;
        std::vector<uint64_t> sel;
        std::vector<int32_t> idx;
        std::vector<uint8_t> acc;
        uint32_t rounds = 0;
        while (!pending.empty() && rounds <= n + 1) {
            const uint64_t m = pending.size();
            rc_.resize(m);
            rm_.resize(m);
            sel.resize(m * W);
            idx.resize(m);
            score.resize(m);
            acc.resize(m);
            for (uint64_t k = 0; k < m; k++) {
                const uint64_t p = pending[k];
                rc_[k] = pods->req_cpu[p];
                rm_[k] = pods->req_mem[p];
                for (uint32_t w = 0; w < W; w++) sel[k * W + w] = pods->sel[p * W + w];
            }
            ks_pods kp{m, rc_.data(), rm_.data(), sel.data(), KS_MEM_HOST};
            ks_bindings kb{idx.data(), score.data(), nullptr, KS_MEM_HOST, nullptr, 0, KS_MEM_HOST, nullptr, nullptr};
            rc = ks_select(s, &kp, policy, KS_SELECT_FORCE_DIRECT, &kb, nullptr); // claims against the current free[]
            if (rc) return rc;
            rc = ks_snapshot_commit_claims(s, m, idx.data(), rc_.data(), rm_.data(), acc.data());
            if (rc) return rc;
            std::vector<uint64_t> next;
            for (uint64_t k = 0; k < m; k++) {
                if (idx[k] < 0) continue; // no feasible node: NoNodeFound (src/main.rs:116-118)
                if (acc[k]) {
                    out_node_idx[pending[k]] = idx[k];
                    if (out_score) out_score[pending[k]] = score[k];
                } else {
                    next.push_back(pending[k]); // lost the node to an earlier pod of the batch: retry
                }
            }
            pending.swap(next);
            rounds++;
        }
        if (out_rounds) *out_rounds = rounds;
        return KS_OK;
    } catch (...) {
        return fail(KS_ERR_NOMEM, "out of host memory in ks_stream_bind");
    }
}

// ---------------------------------------------------------------------------------------------- async streaming
struct StreamItem {
    uint64_t ticket;
    int64_t rc, rm;
    uint64_t sel[KS_MAX_LABEL_WORDS];
};
struct StreamDone {
    uint64_t ticket;
    int32_t node;
    int64_t score;
};
struct ks_stream {
    ks_snapshot* snap = nullptr;
    int policy = KS_SCORE_LEFTOVER;
    uint32_t max_batch = STREAM_BATCH_MAX, W = 1;
    std::mutex mu;
    std::condition_variable cv_work, cv_idle;
    std::deque<StreamItem> in;
    std::deque<StreamDone> out;
    uint64_t submitted = 0, finished = 0, batches = 0, rounds = 0, max_seen = 0;
    bool stop = false;
    bool dead = false; // the dispatcher thread could not start working (out of memory)
    int error = KS_OK;
    std::thread worker;
};

static void stream_worker(ks_stream* q) {
    std::vector<int64_t> rc, rm, score;
    std::vector<uint64_t> sel, tickets;
    std::vector<int32_t> idx;
    try { // every per-batch resize below stays within these capacities: the loop itself never allocates
        rc.reserve(q->max_batch);
        rm.reserve(q->max_batch);
        score.reserve(q->max_batch);
        idx.reserve(q->max_batch);
        tickets.reserve(q->max_batch);
        sel.reserve((size_t)q->max_batch * q->W);
    } catch (...) { // no dispatcher: submissions are answered with the error code by ks_stream_poll / ks_stream_flush
        std::lock_guard<std::mutex> lk(q->mu);
        q->error = KS_ERR_NOMEM;
        q->dead = true;
        q->cv_idle.notify_all();
        return;
    }
    for (;;) {
        {
            std::unique_lock<std::mutex> lk(q->mu);
            q->cv_work.wait(lk, [&] { return q->stop || !q->in.empty(); });
            if (q->stop) return;
            const size_t m = std::min<size_t>(q->in.size(), q->max_batch);
            rc.resize(m);
            rm.resize(m);
            sel.resize(m * q->W);
            tickets.resize(m);
            for (size_t k = 0; k < m; k++) { // everything that has arrived, in arrival order
                const StreamItem& it = q->in.front();
                rc[k] = it.rc;
                rm[k] = it.rm;
                tickets[k] = it.ticket;
                for (uint32_t w = 0; w < q->W; w++) sel[k * q->W + w] = it.sel[w];
                q->in.pop_front();
            }
        }
        const size_t m = rc.size();
        idx.assign(m, -1);
        score.assign(m, 0);
        uint32_t rounds = 0;
        ks_pods kp{m, rc.data(), rm.data(), sel.data(), KS_MEM_HOST};
        const int e = ks_stream_bind(q->snap, &kp, q->policy, idx.data(), score.data(), &rounds);
        {
            std::lock_guard<std::mutex> lk(q->mu);
            if (e) q->error = e;
            try {
                for (size_t k = 0; k < m; k++) q->out.push_back(StreamDone{tickets[k], e ? -1 : idx[k], e ? 0 : score[k]});
            } catch (...) { // results that could not be queued are lost; the poller gets the error code
                q->error = KS_ERR_NOMEM;
            }
            q->finished += m;
            q->batches++;
            q->rounds += rounds;
            q->max_seen = std::max<uint64_t>(q->max_seen, m);
        }
        q->cv_idle.notify_all();
    }
}

int ks_stream_open(ks_snapshot* s, int policy, uint32_t max_batch, ks_stream** out) {
    if (!s || !out) return fail(KS_ERR_INVALID, "NULL argument");
    if (policy != KS_SCORE_LEFTOVER && policy != KS_SCORE_LEAST_ALLOCATED) return fail(KS_ERR_INVALID, "bad policy");
    ks_stream* q = new (std::nothrow) ks_stream();
    if (!q) return fail(KS_ERR_NOMEM, "out of host memory");
    q->snap = s;
    q->policy = policy;
    q->W = s->W;
    q->max_batch = max_batch == 0 ? STREAM_BATCH_MAX : std::min<uint32_t>(max_batch, STREAM_BATCH_MAX);
    try {
        q->worker = std::thread(stream_worker, q);
    } catch (...) {
        delete q;
        return fail(KS_ERR_NOMEM, "cannot start the dispatcher thread");
    }
    *out = q;
    return KS_OK;
}

int ks_stream_submit(ks_stream* q, uint64_t n, const int64_t* req_cpu, const int64_t* req_mem, const uint64_t* sel,
                     const uint64_t* tickets) {
    if (!q || (n && (!req_cpu || !req_mem || !sel || !tickets))) return fail(KS_ERR_INVALID, "NULL argument");
    if (n == 0) return KS_OK;
    try {
        std::lock_guard<std::mutex> lk(q->mu);
        for (uint64_t i = 0; i < n; i++) {
            StreamItem it;
            it.ticket = tickets[i];
            it.rc = req_cpu[i];
            it.rm = req_mem[i];
            for (uint32_t w = 0; w < q->W; w++) it.sel[w] = sel[i * q->W + w];
            q->in.push_back(it);
        }
        q->submitted += n;
    } catch (...) {
        return fail(KS_ERR_NOMEM, "out of host memory");
    }
    q->cv_work.notify_one();
    return KS_OK;
}

int ks_stream_poll(ks_stream* q, uint64_t max, uint64_t* out_ticket, int32_t* out_node_idx, int64_t* out_score, uint64_t* out_n) {
    if (!q || !out_n || (max && (!out_ticket || !out_node_idx))) return fail(KS_ERR_INVALID, "NULL argument");
    std::lock_guard<std::mutex> lk(q->mu);
    uint64_t k = 0;
    while (k < max && !q->out.empty()) {
        const StreamDone& d = q->out.front();
        out_ticket[k] = d.ticket;
        out_node_idx[k] = d.node;
        if (out_score) out_score[k] = d.score;
        q->out.pop_front();
        k++;
    }
    *out_n = k;
    if (q->error) {
        const int e = q->error;
        q->error = KS_OK;
        return e; // ks_last_error() of the dispatcher thread is not visible here: the code says what failed
    }
    return KS_OK;
}

int ks_stream_flush(ks_stream* q) {
    if (!q) return fail(KS_ERR_INVALID, "NULL argument");
    std::unique_lock<std::mutex> lk(q->mu);
    q->cv_idle.wait(lk, [&] { return q->dead || q->finished == q->submitted; });
    if (q->dead) return fail(KS_ERR_NOMEM, "the stream's dispatcher thread is not running (out of host memory)");
    return KS_OK;
}

int ks_stream_stats(ks_stream* q, uint64_t* batches, uint64_t* rounds, uint64_t* max_batch_seen) {
    if (!q) return fail(KS_ERR_INVALID, "NULL argument");
    std::lock_guard<std::mutex> lk(q->mu);
    if (batches) *batches = q->batches;
    if (rounds) *rounds = q->rounds;
    if (max_batch_seen) *max_batch_seen = q->max_seen;
    return KS_OK;
}

void ks_stream_close(ks_stream* q) {
    if (!q) return;
    {
        std::lock_guard<std::mutex> lk(q->mu);
        q->stop = true;
    }
    q->cv_work.notify_all();
    if (q->worker.joinable()) q->worker.join();
    delete q;
}

} // extern "C"
