// Host-side objects behind the C-ABI (include/evstore_b200.h).
#pragma once
#include <cuda_runtime.h>

#include <cstdint>
#include <string>
#include <vector>

#include "../../include/evstore_b200.h"
#include "evs_types.cuh"

namespace evs {

void set_error(const std::string &msg);

#define EVS_CUDA(call)                                                                              \
    do {                                                                                            \
        cudaError_t e__ = (call);                                                                   \
        if (e__ != cudaSuccess) {                                                                   \
            ::evs::set_error(std::string(#call) + " -> " + cudaGetErrorString(e__) + " (" + __FILE__ + ":" + \
                             std::to_string(__LINE__) + ")");                                       \
            return EVS_ERR_CUDA;                                                                    \
        }                                                                                           \
    } while (0)

// Capacities in entries, following the reference's constructors (see evs_api.cu:compute_caps).
struct Caps {
    long long c1 = 0, c2 = 0, c3 = 0;
};
int compute_caps(const evs_config &cfg, Caps &out);

struct Tier {
    TierDev dev{};
    int prec = 0;
    std::vector<void *> allocs;              // device allocations to free
    std::vector<const unsigned char *> store_dev;   // per table, device-visible backing rows
};


// Kernel ids for the launch counter / per-kernel CUDA-event timing (evs_set_profiling).
enum KernelId { K_SERVE = 0, K_SCAN, K_UPDATE, K_EVICT, K_PREFETCH, K_COMPACT, K_PROBE, K_INTERACT, K_GATHER, K_BAGS, K_UPDATE_ROWS, K_STATE, K_COUNT };
static const char *const kKernelNames[K_COUNT] = {"k_serve", "k_scan", "k_update", "k_evict", "k_prefetch", "k_compact", "k_probe", "k_interact",
                                                  "k_gather", "k_bags", "k_update_rows", "k_state"};

struct Profiler {
    bool on = false;
    unsigned long long launches[K_COUNT] = {};
    double ms[K_COUNT] = {};
    unsigned long long timed[K_COUNT] = {};
    struct Rec { int id; cudaEvent_t a, b; };
    std::vector<Rec> pending;
    std::vector<cudaEvent_t> pool;
    cudaEvent_t get() {
        if (!pool.empty()) { cudaEvent_t e = pool.back(); pool.pop_back(); return e; }
        cudaEvent_t e; cudaEventCreate(&e); return e;
    }
    void drain() {
        for (auto &r : pending) {
            cudaEventSynchronize(r.b);
            float t = 0.f;
            if (cudaEventElapsedTime(&t, r.a, r.b) == cudaSuccess) { ms[r.id] += t; timed[r.id]++; }
            pool.push_back(r.a); pool.push_back(r.b);
        }
        pending.clear();
    }
    void destroy() {
        drain();
        for (cudaEvent_t e : pool) cudaEventDestroy(e);
        pool.clear();
    }
};

// Brackets one kernel launch: counts it and, when profiling is on, times it with CUDA events on
// the launching stream.
struct LaunchScope {
    Profiler &p; int id; cudaStream_t st; cudaEvent_t a = nullptr;
    LaunchScope(Profiler &p_, int id_, cudaStream_t st_) : p(p_), id(id_), st(st_) {
        p.launches[id]++;
        if (p.on) { a = p.get(); cudaEventRecord(a, st); }
    }
    ~LaunchScope() {
        if (a) {
            cudaEvent_t b = p.get();
            cudaEventRecord(b, st);
            p.pending.push_back({id, a, b});
            if (p.pending.size() >= 8192) p.drain();
        }
    }
};

// The look-ahead announcement (evs_prefetch): k_prefetch staged, or is staging, the misses of batch number `seq` on the
// indices `idx` of B samples and tags their rows with generation `gen`.  Every announcement draws a new generation
// (next_pf_gen), so the rows of a cancelled or superseded one never match a later batch.
struct Announcement {
    uint64_t seq = 0;                        // 0: none (batch numbers start at 1)
    const void *idx = nullptr;
    int B = 0;
    uint32_t gen = 0;
    bool matches(uint64_t s, const void *i, int b) const { return seq == s && idx == i && B == b; }
    void record(uint64_t s, const void *i, int b) { seq = s, idx = i, B = b; }
    void cancel() { record(0, nullptr, 0); }
};

}  // namespace evs

struct evs_handle_s {
    evs_config cfg{};
    std::vector<int64_t> rows;
    std::vector<int> table_ids;              // global id of local table t
    int n_tiers = 0;
    bool c3_active = false;
    evs::Caps caps;
    evs::Tier tier[EVS_MAX_TIERS];
    evs::Params params{};                    // kernel parameter block (device pointers inside)
    std::vector<void *> c3_allocs;
    cudaStream_t stream = nullptr;           // the handle's own stream
    cudaGraphNode_t serve_node = nullptr;    // its BatchArgs parameter is rewritten before every graph launch
    cudaGraph_t graph_src = nullptr;
    cudaGraphExec_t graph = nullptr;         // k_serve -> [k_scan ->] k_update -> k_evict (eviction + miss-fetch roles)
    // evs_lookup_batches: kGroup consecutive batches captured in one graph
    static constexpr int kGroup = 4;
    int group = 1;
    cudaGraph_t ggraph_src = nullptr;
    cudaGraphExec_t ggraph = nullptr;
    cudaGraphNode_t gserve[kGroup] = {};
    bool use_graph = true;
    bool use_pdl = true;                     // the batch's kernels are chained by programmatic dependent launch
    int fetch_list_ctas = 8;                 // CTAs of the miss-fetch role (EVSTORE_B200_FETCH_LIST_CTAS overrides)
    int evict_ctas = evs::kTierCtas;         // CTAs of k_evict per tier (EVSTORE_B200_EVICT_CTAS overrides)
    // look-ahead (evs_prefetch): k_prefetch for batch seq+1 runs on pf_stream under the kernels of batch seq
    cudaStream_t pf_stream = nullptr;
    cudaEvent_t ev_done[2] = {};             // batch of that parity has finished (its staging rows may be overwritten)
    bool ev_done_valid[2] = {};
    cudaEvent_t ev_pf_ready = nullptr;       // scratch: orders pf_stream after a caller-supplied stream position
    bool pf_ok = false;                      // staging possible (every backing row 16-byte aligned)
    int pf_ctas = 16;
    int pf_mode = 0, pf_wait_mode = 0;       // experiment switches (EVSTORE_B200_PF_MODE / _PF_WAIT)
    uint64_t seq = 0;                        // batches started on this handle
    evs::Announcement pf;                    // the batch the last look-ahead staged for
    unsigned *err_host = nullptr;            // pinned, device-mapped: last device-side error code (0 = none)
    unsigned long long *ring_host = nullptr; // same block: per tier, batch number << 32 | longest ring window after that batch
    int sticky_error = 0;                    // first error evs_check saw
    size_t hbm_bytes = 0;                    // device memory this handle allocated
    evs::GlobalCtl *g = nullptr;             // device
    evs::BatchArgs *d_args = nullptr;        // device copy of the per-batch arguments
    long long *d_rows = nullptr;
    uint8_t *d_agg = nullptr;                // [max_batch]
    // evs_lookup_bags / evs_shard_lookup_bags: the batch's slices (allocated on first use): indices [T][B*P],
    // rows [B*P][bag_cols][D] (bag_cols = T, or n_tables_total on a rank of a sharded cache), hit codes [B*P][T]
    long long *bag_idx = nullptr;
    float *bag_rows = nullptr;
    uint8_t *bag_hit = nullptr;
    int bag_cols = 0;
    // evs_update_rows: scratch hash of one call's keys (grown, synchronously, when a call brings more keys)
    unsigned long long *upd_key = nullptr;
    long long *upd_pos = nullptr;
    size_t upd_cap = 0;                      // entries of each (a power of two, >= 2 n)
    cudaEvent_t ev_upd = nullptr;            // after the last update or state load: orders the look-ahead stream behind it
    // evs_save_state / evs_load_state / evs_dump_*: staging of a snapshot's body behind kStateMetaWords words (grown, synchronously)
    unsigned long long *state_buf = nullptr;
    size_t state_words = 0;
    // staging for the host-buffer paths: slot 0 serves the synchronous call, all kPipeSlots the
    // pipelined one (H2D of batch n+1 and D2H of batch n-1 overlap the kernels of batch n)
    static constexpr int kPipeSlots = 4;
    long long *d_idx[kPipeSlots] = {};
    float *d_out[kPipeSlots] = {};
    uint8_t *d_hit[kPipeSlots] = {};
    cudaStream_t s_in = nullptr, s_out = nullptr;
    cudaEvent_t ev_in[kPipeSlots] = {}, ev_comp[kPipeSlots] = {}, ev_out[kPipeSlots] = {};
    int64_t submitted = 0;
    bool sharded = false;                    // an evs_shard is connected: k_serve<.., true>, k_evict closes the batch with the peers
    std::vector<void *> registered;          // host ranges we page-locked
    int n_ranges = 0, n_ranges_managed = 0;  // host ranges mapped / of them evs_host_alloc (managed) memory
    std::vector<void *> dev_allocs;
    uint64_t batches = 0;
    evs::Profiler prof;
};

// Table-wise sharding over peer memory (evs_shard_*).
struct evs_shard_s {
    evs_handle h = nullptr;
    int rank = 0, world = 1;
    static constexpr unsigned kRecvBufs = 4; // receive buffers: batch e lands in buffer e % 4 of every rank (a group of 4 batches is one graph)
    int batch_max = 0;                       // global batch
    int t_total = 0;
    unsigned char *block = nullptr;          // our exchange block (cudaMalloc, exported by CUDA IPC)
    size_t bytes = 0, off_recv = 0, off_parts = 0, off_oflags = 0, recv_bytes = 0;
    bool fused = true;                       // one-pass exchange inside k_serve (else a separate probe_only pass)
    unsigned char *peer[evs::kMaxPeers] = {};   // peer r's block in our address space (ours at [rank])
    bool opened[evs::kMaxPeers] = {};
    unsigned epoch = 0;
};
