// C-ABI implementation (include/evstore_b200.h): handle life cycle, per-batch kernel
// sequence, host-buffer path, stats / introspection, legacy libcachemanager.so symbols.
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "evs_host.h"
#include "evs_gather.cuh"
#include "evs_interact.cuh"
#include "evs_kernels.cuh"
#include "evs_c3.cuh"
#include "evs_update.cuh"
#include "evs_prefetch.cuh"
#include "evs_bags.cuh"
#include "evs_knn.cuh"
#include "evs_refresh.cuh"
#include "evs_state.cuh"

namespace evs {

static thread_local std::string g_last_error;
void set_error(const std::string &msg) { g_last_error = msg; }

static unsigned next_pow2(unsigned long long v) {
    unsigned long long p = 1;
    while (p < v) p <<= 1;
    return static_cast<unsigned>(p);
}

// Entry capacities exactly as the reference's constructors compute them, quirks included:
//   cache_manager.cpp:22-52   cacheSize = TOTAL_SIZE, TOTAL_SIZE/2 (2 layers); main 16 -> *2, main 4 -> *8,
//                             main 8 gets TOTAL_SIZE and splits inside its constructor
//   evlfu_32.cpp:99-105       C2 of a 32-bit C1: 16 -> cap*2, 8 -> EVLFU_8BIT(cap*4), 4 -> cap*8
//   evlfu_16.cpp:93-98        C2 of a 16-bit C1: 8 -> EVLFU_8BIT(cap*2), 4 -> cap*4
//   evlfu_8.cpp:57-95         EVLFU_8BIT(total): 1 layer total*4; 2 layers total/2*4 and total/2*8;
//                             3 layers (p*total/100)*4, *8, *36 or total/3*4, *8, *36
//     -> an 8-bit C2 is constructed through that same constructor, so it is multiplied by 4 twice.
//   The literal 36 is EV_DIMENSION (one fp32 row holds EV_DIMENSION 4-byte alt keys); we use cfg.dim.
int compute_caps(const evs_config &cfg, Caps &out) {
    const long long total = cfg.total_size;
    const int mp = cfg.main_precision, sp = cfg.secondary_precision;
    if (total <= 0) return EVS_ERR_INVALID;
    auto prec_ok = [](int p) { return p == 32 || p == 16 || p == 8 || p == 4; };
    if (!prec_ok(mp)) return EVS_ERR_INVALID;
    out = Caps();
    if (cfg.n_layers == 1) {
        out.c1 = total * (32 / mp);
        return EVS_OK;
    }
    if (!prec_ok(sp) || sp >= mp) return EVS_ERR_INVALID;
    if (cfg.n_layers == 2) {
        const long long cs = total / 2;
        if (mp == 32) {
            out.c1 = cs;
            out.c2 = (sp == 16) ? cs * 2 : (sp == 8) ? cs * 4 * 4 : cs * 8;
        } else if (mp == 16) {
            out.c1 = cs * 2;
            out.c2 = (sp == 8) ? out.c1 * 2 * 4 : out.c1 * 4;
        } else if (mp == 8) {
            out.c1 = cs * 4;
            out.c2 = cs * 8;
        } else {
            return EVS_ERR_INVALID;
        }
        return EVS_OK;
    }
    if (cfg.n_layers == 3) {
        if (mp != 8 || sp != 4) return EVS_ERR_INVALID;      // cache_manager.cpp:212-220
        if (cfg.prop_c1 || cfg.prop_c2 || cfg.prop_c3) {
            if (cfg.prop_c1 + cfg.prop_c2 + cfg.prop_c3 != 100) return EVS_ERR_INVALID;
            out.c1 = (cfg.prop_c1 * total / 100) * 4;
            out.c2 = (cfg.prop_c2 * total / 100) * 8;
            out.c3 = (cfg.prop_c3 * total / 100) * cfg.dim;
        } else {
            out.c1 = total / 3 * 4;
            out.c2 = total / 3 * 8;
            out.c3 = total / 3 * cfg.dim;
        }
        return EVS_OK;
    }
    return EVS_ERR_INVALID;
}

// Entry points that launch or copy run under the handle's device whatever the caller's current device is
// (one process may drive several GPUs; torch's current device need not be cfg.device), and restore it.
struct DeviceGuard {
    int prev = -1;
    bool switched = false;
    explicit DeviceGuard(int dev) {
        if (cudaGetDevice(&prev) == cudaSuccess && prev != dev) switched = cudaSetDevice(dev) == cudaSuccess;
    }
    ~DeviceGuard() {
        if (switched) cudaSetDevice(prev);
    }
};

static thread_local size_t *t_alloc_bytes = nullptr;     // evs_create / pipe_init: device bytes are added to the handle's count

template <typename T>
static int dev_alloc(std::vector<void *> &owner, T **p, size_t n, bool zero = true) {
    void *q = nullptr;
    const size_t bytes = std::max<size_t>(n, 1) * sizeof(T);
    EVS_CUDA(cudaMalloc(&q, bytes));
    if (t_alloc_bytes) *t_alloc_bytes += bytes;
    owner.push_back(q);
    if (zero) EVS_CUDA(cudaMemset(q, 0, bytes));
    *p = static_cast<T *>(q);
    return EVS_OK;
}

// Device-visible alias of a host range: ranges that are already page-locked by somebody else (cudaHostAlloc /
// a framework's pinned allocator) are used as they are; anything else is page-locked and mapped here.  Ranges WE
// page-locked live in a process-wide, reference-counted registry: handles normally share backing arrays (EvStore
// passes the caller's fp32 tables through uncopied, and the legacy store plus an EvStore over the same tables is
// a usual setup), so a range is unregistered only when the last handle that maps it is destroyed.
// Lifetime rule for the caller: the host range must outlive every handle created over it.
struct HostReg {
    size_t bytes;
    int refs;
};
static std::mutex g_reg_mu;
static std::map<void *, HostReg> g_reg;

static int map_host_range(evs_handle h, void *hp, size_t bytes, void **dp, const std::string &what) {
    std::lock_guard<std::mutex> lk(g_reg_mu);
    h->n_ranges++;
    auto it = g_reg.find(hp);
    if (it != g_reg.end() && it->second.bytes >= bytes) {
        it->second.refs++;
        h->registered.push_back(hp);
    } else {
        cudaPointerAttributes attr{};
        cudaError_t e = cudaPointerGetAttributes(&attr, hp);
        if (e != cudaSuccess) cudaGetLastError();
        if (e == cudaSuccess && attr.type == cudaMemoryTypeManaged) {
            // evs_host_alloc memory (managed, resident in host memory, mapped into the device): the same address on both sides
            *dp = hp;
            h->n_ranges_managed++;
            return EVS_OK;
        }
        if (e != cudaSuccess || attr.type != cudaMemoryTypeHost) {
            e = cudaHostRegister(hp, bytes, cudaHostRegisterMapped | cudaHostRegisterPortable);
            if (e == cudaSuccess) {
                g_reg[hp] = HostReg{bytes, 1};
                h->registered.push_back(hp);
            } else if (e == cudaErrorHostMemoryAlreadyRegistered) {
                cudaGetLastError();
            } else {
                set_error("cudaHostRegister(" + what + ", " + std::to_string(bytes) + " B) -> " + cudaGetErrorString(e));
                cudaGetLastError();
                return EVS_ERR_CUDA;
            }
        }
    }
    EVS_CUDA(cudaHostGetDevicePointer(dp, hp, 0));
    return EVS_OK;
}

static void release_host_ranges(evs_handle h) {
    std::lock_guard<std::mutex> lk(g_reg_mu);
    for (void *p : h->registered) {
        auto it = g_reg.find(p);
        if (it == g_reg.end()) continue;
        if (--it->second.refs == 0) {
            cudaHostUnregister(p);
            g_reg.erase(it);
        }
    }
    h->registered.clear();
}

static int make_store(evs_handle h, const void *const *ptrs, int prec, std::vector<const unsigned char *> &out) {
    const evs_config &c = h->cfg;
    out.clear();
    for (int t = 0; t < c.n_tables; ++t) {
        const size_t bytes = static_cast<size_t>(h->rows[t]) * c.dim * prec / 8;
        if (ptrs == nullptr || ptrs[t] == nullptr) {
            set_error("backing store pointer missing for table " + std::to_string(t));
            return EVS_ERR_INVALID;
        }
        if (c.store_in_hbm) {
            unsigned char *d = nullptr;
            int rc = dev_alloc(h->dev_allocs, &d, bytes + 16, false);
            if (rc) return rc;
            EVS_CUDA(cudaMemcpy(d, ptrs[t], bytes, cudaMemcpyHostToDevice));
            out.push_back(d);
        } else {
            void *hp = const_cast<void *>(ptrs[t]);
            void *dp = nullptr;
            int rc2 = map_host_range(h, hp, bytes, &dp, "table " + std::to_string(t));
            if (rc2) return rc2;
            out.push_back(static_cast<const unsigned char *>(dp));
        }
    }
    return EVS_OK;
}

static int build_tier(evs_handle h, Tier &tr, int prec, long long cap, const void *const *store) {
    const evs_config &c = h->cfg;
    const long long n_max = static_cast<long long>(c.max_batch) * c.n_tables;
    if (cap < 32) {
        set_error("tier capacity below 32 entries");
        return EVS_ERR_INVALID;
    }
    // the index holds cap entries between batches and up to cap + n_max while a batch is in flight
    // load factor <= 1/3: linear-probing clusters stay short, which bounds the dependent-access
    // chains of probes, claims and evictions (the slab is slot-indexed, so this is also its size)
    const unsigned long long want_slots = static_cast<unsigned long long>(cap + n_max) * 3ull;
    if (want_slots >= (1ull << 31)) {
        set_error("tier too large: the index must stay below 2^31 slots");
        return EVS_ERR_INVALID;
    }
    TierDev &d = tr.dev;
    tr.prec = prec;
    d.prec = prec;
    d.cap = static_cast<unsigned>(cap);
    d.row_bytes = static_cast<unsigned>(c.dim * prec / 8);
    d.row_stride = (d.row_bytes + 15u) & ~15u;
    // the defaults are the reference's *double* constants (evlfu_32.hpp:53-54): int(cap * 0.95) with 0.95f
    // widened to double is one less for cap = 60
    const double pic = c.perfect_item_cap > 0 ? static_cast<double>(c.perfect_item_cap) : 0.95;
    const double fr = c.flush_rate > 0 ? static_cast<double>(c.flush_rate) : 0.3;
    d.max_perfect = static_cast<unsigned>(static_cast<int>(static_cast<double>(cap) * pic));
    d.flush_n = static_cast<unsigned>(static_cast<int>(fr * static_cast<double>(cap))) + 1u;
    d.n_buckets = c.n_tables_total + 1;
    const unsigned hash_cap = next_pow2(want_slots);
    d.hash_mask = hash_cap - 1;
    // room for the live entries plus 64 batches of appends: the host may run that far ahead of the device before it has to
    // wait for the ring mirror to advance (maintain_rings)
    long long slack = 64;
    if (const char *rs = getenv("EVSTORE_B200_RING_SLACK"))         // testing aid: small rings, so that compaction runs within a few batches
        if (atoi(rs) >= 5) slack = atoi(rs);
    d.ring_cap = next_pow2(static_cast<unsigned long long>(std::max(2 * (cap + n_max), cap + slack * n_max)));
    int rc;
    if ((rc = dev_alloc(tr.allocs, &d.slots, hash_cap, false))) return rc;
    if ((rc = dev_alloc(tr.allocs, &d.slab, static_cast<size_t>(hash_cap) * d.row_stride, true))) return rc;
    if ((rc = dev_alloc(tr.allocs, &d.ring, static_cast<size_t>(d.n_buckets) * d.ring_cap, false))) return rc;
    if ((rc = dev_alloc(tr.allocs, &d.ctl, 1, true))) return rc;
    if ((rc = dev_alloc(tr.allocs, &d.evicted, n_max, true))) return rc;
    // one look-back entry per eviction chunk; the records of all rings bound the number of chunks
    d.lb_cap = static_cast<unsigned>(static_cast<unsigned long long>(d.n_buckets) * d.ring_cap / kEvictWindow + d.n_buckets + 64);
    if ((rc = dev_alloc(tr.allocs, &d.lookback, d.lb_cap, true))) return rc;
    d.flushed = nullptr;
    if (c.record_events)
        if ((rc = dev_alloc(tr.allocs, &d.flushed, d.flush_n, true))) return rc;

    if ((rc = make_store(h, store, prec, tr.store_dev))) return rc;
    const unsigned char **dstore = nullptr;
    if ((rc = dev_alloc(tr.allocs, &dstore, c.n_tables, false))) return rc;
    EVS_CUDA(cudaMemcpy(dstore, tr.store_dev.data(), sizeof(void *) * c.n_tables, cudaMemcpyHostToDevice));
    d.store = dstore;

    k_init_tier<<<592, 256, 0, h->stream>>>(d);
    EVS_CUDA(cudaGetLastError());
    EVS_CUDA(cudaStreamSynchronize(h->stream));
    return EVS_OK;
}

static int build_c3(evs_handle h) {
    const evs_config &c = h->cfg;
    C3Dev &d = h->params.c3;
    const long long n_max = static_cast<long long>(c.max_batch) * c.n_tables;
    const long long cap = h->caps.c3;
    if (c.alt_keys == nullptr) {
        set_error("n_layers == 3 needs alt_keys");
        return EVS_ERR_INVALID;
    }
    d.cap = static_cast<unsigned>(cap);
    const unsigned hash_cap = next_pow2(static_cast<unsigned long long>(cap + 2 * n_max) * 3ull / 2ull);
    d.hash_mask = hash_cap - 1;
    d.ring_cap = next_pow2(static_cast<unsigned long long>(4 * cap + 8 * n_max));
    int rc;
    if ((rc = dev_alloc(h->c3_allocs, &d.slots, hash_cap, false))) return rc;
    if ((rc = dev_alloc(h->c3_allocs, &d.scratch, hash_cap, false))) return rc;
    if ((rc = dev_alloc(h->c3_allocs, &d.ring, d.ring_cap, true))) return rc;
    if ((rc = dev_alloc(h->c3_allocs, &d.ctl, 1, true))) return rc;
    // alt-key tables: device-visible like the backing store
    std::vector<const unsigned int *> ptrs;
    for (int t = 0; t < c.n_tables; ++t) {
        const size_t bytes = static_cast<size_t>(h->rows[t]) * sizeof(uint32_t);
        if (c.alt_keys[t] == nullptr) {
            set_error("alt_keys pointer missing for table " + std::to_string(t));
            return EVS_ERR_INVALID;
        }
        if (c.store_in_hbm) {
            unsigned int *dp = nullptr;
            if ((rc = dev_alloc(h->c3_allocs, &dp, h->rows[t], false))) return rc;
            EVS_CUDA(cudaMemcpy(dp, c.alt_keys[t], bytes, cudaMemcpyHostToDevice));
            ptrs.push_back(dp);
        } else {
            void *hp = const_cast<uint32_t *>(c.alt_keys[t]);
            void *dp = nullptr;
            if ((rc = map_host_range(h, hp, bytes, &dp, "alt keys " + std::to_string(t)))) return rc;
            ptrs.push_back(static_cast<const unsigned int *>(dp));
        }
    }
    const unsigned int **dalt = nullptr;
    if ((rc = dev_alloc(h->c3_allocs, &dalt, c.n_tables, false))) return rc;
    EVS_CUDA(cudaMemcpy(dalt, ptrs.data(), sizeof(void *) * c.n_tables, cudaMemcpyHostToDevice));
    d.alt = dalt;
    d.active = 1;
    k_init_c3<<<592, 256, 0, h->stream>>>(d);
    EVS_CUDA(cudaGetLastError());
    EVS_CUDA(cudaStreamSynchronize(h->stream));
    return EVS_OK;
}

static void destroy_graphs(evs_handle h);
static void free_all(evs_handle h) {
    if (h == nullptr) return;
    cudaSetDevice(h->cfg.device);
    cudaDeviceSynchronize();
    destroy_graphs(h);
    for (int i = 0; i < EVS_MAX_TIERS; ++i)
        for (void *p : h->tier[i].allocs) cudaFree(p);
    for (void *p : h->c3_allocs) cudaFree(p);
    for (void *p : h->dev_allocs) cudaFree(p);
    if (h->upd_key) cudaFree(h->upd_key);
    if (h->upd_pos) cudaFree(h->upd_pos);
    if (h->ev_upd) cudaEventDestroy(h->ev_upd);
    if (h->state_buf) cudaFree(h->state_buf);
    release_host_ranges(h);
    h->prof.destroy();
    if (h->pf_stream) cudaStreamDestroy(h->pf_stream);
    for (int i = 0; i < 2; ++i)
        if (h->ev_done[i]) cudaEventDestroy(h->ev_done[i]);
    if (h->ev_pf_ready) cudaEventDestroy(h->ev_pf_ready);
    if (h->err_host) cudaFreeHost(h->err_host);
    if (h->s_in) cudaStreamDestroy(h->s_in);
    if (h->s_out) cudaStreamDestroy(h->s_out);
    for (int i = 0; i < evs_handle_s::kPipeSlots; ++i) {
        if (h->ev_in[i]) cudaEventDestroy(h->ev_in[i]);
        if (h->ev_comp[i]) cudaEventDestroy(h->ev_comp[i]);
        if (h->ev_out[i]) cudaEventDestroy(h->ev_out[i]);
    }
    if (h->stream) cudaStreamDestroy(h->stream);
    cudaGetLastError();
    delete h;
}

// Keep every bucket ring from overflowing.  The last CTA of k_evict mirrors, per tier, the longest ring window
// (max over the buckets of tail - head) together with the batch number into mapped pinned memory, so the host knows the
// occupancy as of the last FINISHED batch without touching the device; every batch started since can append at most
// max_batch * n_tables records.  When that bound gets close to the ring size the host first lets the device catch up
// (bounded run-ahead: it spins on the mirror, the device keeps its queue), and only a ring that is really full is
// compacted (stream synchronise + k_compact).
static bool ring_fits(evs_handle h, int ti, int ahead) {
    const Tier &tr = h->tier[ti];
    const unsigned long long n_max = static_cast<unsigned long long>(h->cfg.max_batch) * h->cfg.n_tables;
    const unsigned long long v = *reinterpret_cast<volatile unsigned long long *>(h->ring_host + ti);
    const unsigned long long used = v & 0xFFFFFFFFull;
    unsigned in_flight = static_cast<unsigned>(h->seq) - static_cast<unsigned>(v >> 32);
    if (static_cast<int>(in_flight) < 0) in_flight = 0;      // replays of a caller's graph not reported yet (evs_note_replays)
    return used + (static_cast<unsigned long long>(in_flight) + ahead) * n_max <= tr.dev.ring_cap;
}

static int maintain_rings(evs_handle h, int ti, cudaStream_t st, int ahead = 2) {
    if (ring_fits(h, ti, ahead)) return EVS_OK;
    Tier &tr = h->tier[ti];
    const unsigned long long n_max = static_cast<unsigned long long>(h->cfg.max_batch) * h->cfg.n_tables;
    // let the device catch up: the mirror advances with every batch that finishes
    {
        unsigned long long spins = 0;
        while (!ring_fits(h, ti, ahead)) {
            const unsigned long long v = *reinterpret_cast<volatile unsigned long long *>(h->ring_host + ti);
            if (static_cast<unsigned>(v >> 32) == static_cast<unsigned>(h->seq)) break;      // nothing in flight: the ring is full
            if (++spins > (1ull << 22)) {                                                    // ~ tens of ms without progress
                if (cudaStreamQuery(st) != cudaErrorNotReady) break;
                spins = 0;
            }
        }
        if (ring_fits(h, ti, ahead)) return EVS_OK;
    }
    TierCtl ctl;
    EVS_CUDA(cudaStreamSynchronize(st));
    EVS_CUDA(cudaMemcpy(&ctl, tr.dev.ctl, sizeof(ctl), cudaMemcpyDeviceToHost));
    bool any = false;
    for (int b = 0; b < tr.dev.n_buckets; ++b) {
        if (ctl.tail[b] - ctl.head[b] + static_cast<unsigned long long>(ahead) * n_max > tr.dev.ring_cap) {
            LaunchScope ls(h->prof, K_COMPACT, st);
            k_compact<<<1, 1024, 0, st>>>(tr.dev, b);
            any = true;
        }
    }
    EVS_CUDA(cudaGetLastError());
    if (any) {
        EVS_CUDA(cudaStreamSynchronize(st));
        EVS_CUDA(cudaMemcpy(&ctl, tr.dev.ctl, sizeof(ctl), cudaMemcpyDeviceToHost));
    }
    unsigned long long mx = 0;
    for (int b = 0; b < tr.dev.n_buckets; ++b) mx = std::max(mx, ctl.tail[b] - ctl.head[b]);
    // the device is idle: the host refreshes the mirror itself
    *reinterpret_cast<volatile unsigned long long *>(h->ring_host + ti) = (static_cast<unsigned long long>(static_cast<unsigned>(h->seq)) << 32) | mx;
    return EVS_OK;
}

// ---- kernel selection by (main precision, secondary precision) -----------------------------
using KernelFn = void (*)(const Params);
using ServeFn = void (*)(const Params, const BatchArgs);
using PrefetchFn = void (*)(const Params, const PrefetchArgs);
using RefreshFn = void (*)(const Params, const RefreshArgs);
struct KernelSet {
    ServeFn serve = nullptr;        // one GPU
    ServeFn serve_sh = nullptr;     // one rank of a table-wise sharded cache
    KernelFn evict = nullptr;       // eviction + miss-fetch roles
    PrefetchFn prefetch = nullptr;
    RefreshFn update_rows = nullptr;   // evs_update_rows (evs_refresh.cuh)
};
template <int P0, int P1>
static KernelSet kernels_of() {
    KernelSet k;
    k.serve = k_serve<P0, P1, false>;
    k.serve_sh = k_serve<P0, P1, true>;
    k.evict = k_evict<P0, P1>;
    k.prefetch = k_prefetch<P0, P1>;
    k.update_rows = k_update_rows<P0, P1>;
    return k;
}
static KernelSet pick_kernels(int p0, int p1) {
    switch (p0 * 100 + p1) {
        case 3200: return kernels_of<32, 0>();
        case 1600: return kernels_of<16, 0>();
        case 800: return kernels_of<8, 0>();
        case 400: return kernels_of<4, 0>();
        case 3216: return kernels_of<32, 16>();
        case 3208: return kernels_of<32, 8>();
        case 3204: return kernels_of<32, 4>();
        case 1608: return kernels_of<16, 8>();
        case 1604: return kernels_of<16, 4>();
        case 804: return kernels_of<8, 4>();
        default: return KernelSet();
    }
}
static KernelSet kernels_of_handle(evs_handle h) { return pick_kernels(h->tier[0].prec, h->n_tiers == 2 ? h->tier[1].prec : 0); }
static ServeFn serve_of(evs_handle h, const KernelSet &ks) { return h->sharded ? ks.serve_sh : ks.serve; }

// A launch; `pdl`: the kernel may start while its predecessor on the stream drains (programmatic stream
// serialization) -- it blocks in griddepcontrol.wait before it touches anything the predecessor wrote.
static cudaError_t launch_ex(const void *fn, dim3 grid, int block, size_t smem, cudaStream_t st, void **args, bool pdl) {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = grid;
    cfg.blockDim = dim3(block);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = pdl ? at : nullptr;
    cfg.numAttrs = pdl ? 1 : 0;
    return cudaLaunchKernelExC(&cfg, fn, args);
}

static cudaError_t launch_serve(ServeFn fn, int grid, cudaStream_t st, const Params &p, const BatchArgs &a, bool pdl = false) {
    void *args[] = {const_cast<Params *>(&p), const_cast<BatchArgs *>(&a)};
    return launch_ex(reinterpret_cast<const void *>(fn), dim3(grid), kLookupThreads, 0, st, args, pdl);
}

static cudaError_t launch(KernelFn fn, dim3 grid, int block, size_t smem, cudaStream_t st, const Params &p, bool pdl) {
    void *args[] = {const_cast<Params *>(&p)};
    return launch_ex(reinterpret_cast<const void *>(fn), grid, block, smem, st, args, pdl);
}

static size_t fetch_smem(evs_handle h) {
    unsigned s = h->tier[0].dev.row_stride;
    if (h->n_tiers == 2) s = std::max(s, h->tier[1].dev.row_stride);
    return static_cast<size_t>(kEvictThreads / 32) * s;
}

// The per-batch kernel sequence, a linear chain on one stream:
//     k_serve -> [k_scan ->] k_update -> k_evict {eviction of each tier || miss fetch}
// (the zero-copy miss fetch used to be its own kernel on a side stream next to k_evict; as a role of k_evict's grid
// the graph has no fork / join, and with evs_prefetch its rows are mostly staged in HBM already).
// `n_chunks` CTAs of k_serve / k_update; CTAs past the batch end exit at once, so a captured graph
// uses the maximum.
static int enqueue_batch(evs_handle h, cudaStream_t st, int n_chunks, const BatchArgs &a, bool serve_pdl) {
    const Params &p = h->params;
    const KernelSet ks = kernels_of_handle(h);
    Profiler &pf = h->prof;
    const bool pdl = h->use_pdl && !pf.on;                // event records between the launches would serialise them anyway
    // serve_pdl: k_serve is a programmatic dependent of the kernel that precedes it -- the previous batch's k_evict, on the
    // stream of a serving loop or inside a graph of several batches (never the first node of a graph)
    { LaunchScope ls(pf, K_SERVE, st); EVS_CUDA(launch_serve(serve_of(h, ks), n_chunks, st, p, a, pdl && serve_pdl)); }
    if (p.n_chunks_max > p.quad_max) {
        LaunchScope ls(pf, K_SCAN, st);
        EVS_CUDA(launch(k_scan, (h->n_tiers == 1 ? 1 : kSeqGroups) * h->tier[0].dev.n_buckets, 256, 0, st, p, pdl));
    }
    { LaunchScope ls(pf, K_UPDATE, st); 
        // a sample per warp (26 tables): per-sample sums of the earlier CTAs' counts; packed warps: one sum per CTA
        KernelFn upd = p.policy == EVS_POLICY_LFU ? k_update<1, 8, true, true>
                       : h->n_tiers == 1 ? (p.L == 32 ? k_update<1, 8, false> : k_update<1, 8, true>)
                                       : (p.L == 32 ? k_update<kSeqGroups, 4, false> : k_update<kSeqGroups, 4, true>);
        EVS_CUDA(launch(upd, n_chunks, kLookupThreads, 0, st, p, pdl)); }
    {
        LaunchScope ls(pf, K_EVICT, st);
        EVS_CUDA(launch(ks.evict, dim3(std::max(h->evict_ctas, h->fetch_list_ctas), h->n_tiers + 1), kEvictThreads, fetch_smem(h), st, p, pdl));
    }
    return EVS_OK;
}

// Capture `nb` consecutive batches into one graph.  Only the BatchArgs parameter of the k_serve nodes changes between
// launches; the nodes are told apart by the marker the capture puts into BatchArgs::seq.
constexpr unsigned kSeqMarker = 0xE5000000u;
static int build_graph_n(evs_handle h, int nb, cudaGraph_t *src_out, cudaGraphExec_t *exec_out, cudaGraphNode_t *serve_nodes) {
    cudaGraph_t g = nullptr;
    const bool was_on = h->prof.on;
    h->prof.on = false;                                   // no event records inside the capture
    unsigned long long saved[K_COUNT];
    memcpy(saved, h->prof.launches, sizeof(saved));
    EVS_CUDA(cudaStreamBeginCapture(h->stream, cudaStreamCaptureModeThreadLocal));
    int rc = EVS_OK;
    for (int i = 0; i < nb && rc == EVS_OK; ++i) {
        BatchArgs none{};
        none.seq = kSeqMarker + static_cast<unsigned>(i);
        rc = enqueue_batch(h, h->stream, h->params.n_chunks_max, none, i > 0);
    }
    cudaError_t e = cudaStreamEndCapture(h->stream, &g);
    memcpy(h->prof.launches, saved, sizeof(saved));
    h->prof.on = was_on;
    if (rc) return rc;
    EVS_CUDA(e);
    size_t n_nodes = 0;
    EVS_CUDA(cudaGraphGetNodes(g, nullptr, &n_nodes));
    std::vector<cudaGraphNode_t> nodes(n_nodes);
    EVS_CUDA(cudaGraphGetNodes(g, nodes.data(), &n_nodes));
    const KernelSet ks = kernels_of_handle(h);
    for (int i = 0; i < nb; ++i) serve_nodes[i] = nullptr;
    for (cudaGraphNode_t nd : nodes) {
        cudaGraphNodeType ty;
        EVS_CUDA(cudaGraphNodeGetType(nd, &ty));
        if (ty != cudaGraphNodeTypeKernel) continue;
        cudaKernelNodeParams kp{};
        EVS_CUDA(cudaGraphKernelNodeGetParams(nd, &kp));
        if (kp.func != reinterpret_cast<void *>(serve_of(h, ks)) || kp.kernelParams == nullptr) continue;
        const unsigned mark = static_cast<const BatchArgs *>(kp.kernelParams[1])->seq - kSeqMarker;
        if (mark < static_cast<unsigned>(nb)) serve_nodes[mark] = nd;
    }
    for (int i = 0; i < nb; ++i)
        if (serve_nodes[i] == nullptr) {
            set_error("graph capture: k_serve node not found");
            cudaGraphDestroy(g);
            return EVS_ERR_CUDA;
        }
    EVS_CUDA(cudaGraphInstantiate(exec_out, g, 0));
    *src_out = g;                                         // kept: the node handles belong to it
    return EVS_OK;
}

static void destroy_graphs(evs_handle h) {
    if (h->graph) cudaGraphExecDestroy(h->graph);
    if (h->graph_src) cudaGraphDestroy(h->graph_src);
    if (h->ggraph) cudaGraphExecDestroy(h->ggraph);
    if (h->ggraph_src) cudaGraphDestroy(h->ggraph_src);
    h->graph = h->ggraph = nullptr;
    h->graph_src = h->ggraph_src = nullptr;
}

// The single-batch graph, and -- for evs_lookup_batches -- one of kGroup batches: a graph-to-graph boundary costs
// ~5 us on the device, a kernel boundary inside a graph (programmatic edge) under 1 us.
static int build_graph(evs_handle h) {
    int rc = build_graph_n(h, 1, &h->graph_src, &h->graph, &h->serve_node);
    if (rc) return rc;
    const char *gg = getenv("EVSTORE_B200_GROUP");        // tuning aid: batches per group graph (1 = none)
    h->group = evs_handle_s::kGroup;
    if (gg && atoi(gg) >= 1) h->group = std::min(atoi(gg), static_cast<int>(evs_handle_s::kGroup));
    if (h->group > 1) {
        rc = build_graph_n(h, h->group, &h->ggraph_src, &h->ggraph, h->gserve);
        if (rc) {                                         // not fatal: batches then go one graph each
            cudaGetLastError();
            h->group = 1;
            h->ggraph = nullptr;
            h->ggraph_src = nullptr;
        }
    }
    return EVS_OK;
}

static int check_device_errors(evs_handle h) {
    GlobalCtl g;
    EVS_CUDA(cudaMemcpy(&g, h->g, sizeof(g), cudaMemcpyDeviceToHost));
    if (g.error) {
        unsigned zero = 0;
        cudaMemcpy(&h->g->error, &zero, sizeof(zero), cudaMemcpyHostToDevice);
        *reinterpret_cast<volatile unsigned *>(h->err_host) = 0u;
        h->sticky_error = 0;
        if (g.error == 7u) {
            set_error("a peer rank did not deliver its hit counts / rows in time (table-wise sharding)");
            return EVS_ERR_PEER;
        }
        set_error("an index was outside [0, rows[table])");
        return EVS_ERR_INDEX;
    }
    for (int i = 0; i < h->n_tiers; ++i) {
        TierCtl c;
        EVS_CUDA(cudaMemcpy(&c, h->tier[i].dev.ctl, sizeof(c), cudaMemcpyDeviceToHost));
        if (c.error) {
            set_error("tier " + std::to_string(i) + ": internal capacity error " + std::to_string(c.error));
            return EVS_ERR_CAPACITY;
        }
    }
    if (h->c3_active) {
        C3Ctl c;
        EVS_CUDA(cudaMemcpy(&c, h->params.c3.ctl, sizeof(c), cudaMemcpyDeviceToHost));
        if (c.error) {
            set_error("C3: internal capacity error " + std::to_string(c.error));
            return EVS_ERR_CAPACITY;
        }
    }
    return EVS_OK;
}

}  // namespace evs

using namespace evs;

extern "C" {

static int poll_error(evs_handle h);

int evs_version(void) { return 100; }

const char *evs_last_error(void) { return g_last_error.c_str(); }

int evs_create(const evs_config *cfg, evs_handle *out) {
    if (cfg == nullptr || out == nullptr) return EVS_ERR_INVALID;
    *out = nullptr;
    if (cfg->n_tables < 1 || cfg->n_tables > EVS_MAX_TABLES || cfg->dim < 1 || cfg->max_batch < 1 ||
        cfg->rows == nullptr || cfg->n_layers < 1 || cfg->n_layers > 3) {
        set_error("evs_create: bad n_tables / dim / max_batch / rows / n_layers");
        return EVS_ERR_INVALID;
    }
    if (static_cast<unsigned long long>(cfg->max_batch) * cfg->n_tables > kMaxProtPositions) {
        set_error("evs_create: max_batch * n_tables must not exceed 2^27 positions");
        return EVS_ERR_INVALID;
    }
    evs_handle h = new evs_handle_s();
    h->cfg = *cfg;
    if (h->cfg.n_tables_total <= 0) h->cfg.n_tables_total = cfg->n_tables;
    if (h->cfg.n_tables_total > 31 || h->cfg.n_tables_total < cfg->n_tables) {
        set_error("evs_create: n_tables_total must be in [n_tables, 31]");
        delete h;
        return EVS_ERR_INVALID;
    }
    // global table ids: keys, the agg_hit buckets and -- sharded -- the peers' receive-buffer columns are derived from
    // them, so an id outside [0, n_tables_total) would alias another table's keys and write outside a peer's buffer
    h->table_ids.resize(cfg->n_tables);
    for (int t = 0; t < cfg->n_tables; ++t) h->table_ids[t] = cfg->table_ids ? cfg->table_ids[t] : cfg->table_base + t;
    h->cfg.table_ids = nullptr;
    for (int t = 0; t < cfg->n_tables; ++t) {
        const int g = h->table_ids[t];
        if (g < 0 || g >= h->cfg.n_tables_total || (t > 0 && g <= h->table_ids[t - 1])) {
            set_error("evs_create: table ids (table_base + t, or table_ids[t]) must be strictly increasing and lie in [0, n_tables_total)");
            delete h;
            return EVS_ERR_INVALID;
        }
    }
    if (h->cfg.high_agghit_threshold <= 0) h->cfg.high_agghit_threshold = 23;
    if (cfg->policy != EVS_POLICY_EVLFU && cfg->policy != EVS_POLICY_LRU && cfg->policy != EVS_POLICY_LFU) {
        set_error("evs_create: unknown policy");
        delete h;
        return EVS_ERR_INVALID;
    }
    if (cfg->policy != EVS_POLICY_EVLFU && (cfg->n_layers != 1 || cfg->approx_emb_thres > 0)) {
        set_error("evs_create: the LRU / LFU policies (cache_algo/LRU.py, LFU.py) are single-layer and have no approximate substitution");
        delete h;
        return EVS_ERR_INVALID;
    }
    if ((static_cast<long long>(cfg->dim) * cfg->main_precision) % 8 != 0) {
        set_error("evs_create: dim*precision must be a whole number of bytes");
        delete h;
        return EVS_ERR_INVALID;
    }
    h->rows.assign(cfg->rows, cfg->rows + cfg->n_tables);
    h->cfg.rows = h->rows.data();
    for (int t = 0; t < cfg->n_tables; ++t) {
        if (h->rows[t] < 1 || h->rows[t] >= (1ll << kKeyShift)) {
            set_error("evs_create: rows[t] out of range");
            delete h;
            return EVS_ERR_INVALID;
        }
    }
    int rc = compute_caps(h->cfg, h->caps);
    if (rc) {
        set_error("evs_create: unsupported layer / precision / size combination");
        delete h;
        return rc;
    }
    cudaError_t e = cudaSetDevice(cfg->device);
    if (e != cudaSuccess) {
        set_error(std::string("cudaSetDevice -> ") + cudaGetErrorString(e));
        delete h;
        return EVS_ERR_CUDA;
    }
    auto fail = [&](int code) {
        free_all(h);
        return code;
    };
    t_alloc_bytes = &h->hbm_bytes;
    struct AllocScope {
        ~AllocScope() { t_alloc_bytes = nullptr; }
    } alloc_scope;
    if (cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaStreamCreateWithFlags(&h->pf_stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreateWithFlags(&h->ev_done[0], cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&h->ev_done[1], cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&h->ev_pf_ready, cudaEventDisableTiming) != cudaSuccess ||
        cudaHostAlloc(reinterpret_cast<void **>(&h->err_host), 256, cudaHostAllocMapped | cudaHostAllocPortable) != cudaSuccess) {
        set_error("cudaStreamCreate / cudaEventCreate / cudaHostAlloc failed");
        return fail(EVS_ERR_CUDA);
    }
    memset(h->err_host, 0, 256);
    h->ring_host = reinterpret_cast<unsigned long long *>(reinterpret_cast<unsigned char *>(h->err_host) + 64);
    h->n_tiers = cfg->n_layers >= 2 ? 2 : 1;
    if (pick_kernels(cfg->main_precision, h->n_tiers == 2 ? cfg->secondary_precision : 0).serve == nullptr) {
        set_error("evs_create: no kernel for this precision pair");
        return fail(EVS_ERR_INVALID);
    }
    if (h->n_tiers == 2 && (static_cast<long long>(cfg->dim) * cfg->secondary_precision) % 8 != 0) {
        set_error("evs_create: dim*secondary_precision must be a whole number of bytes");
        return fail(EVS_ERR_INVALID);
    }
    const long long n_max = static_cast<long long>(cfg->max_batch) * cfg->n_tables;
    int L = 1, L_shift = 0;                 // lanes per sample = next_pow2(n_tables)
    while (L < cfg->n_tables) L <<= 1, ++L_shift;
    const int spc = kSamplesPerCta * (32 / L);
    const int n_chunks_max = (cfg->max_batch + spc - 1) / spc;
    Params &P = h->params;
    if ((rc = dev_alloc(h->dev_allocs, &h->g, 1))) return fail(rc);
    if ((rc = dev_alloc(h->dev_allocs, &h->d_args, 1))) return fail(rc);
    if ((rc = dev_alloc(h->dev_allocs, &h->d_rows, cfg->n_tables))) return fail(rc);
    if (cudaMemcpy(h->d_rows, h->rows.data(), sizeof(int64_t) * cfg->n_tables, cudaMemcpyHostToDevice) != cudaSuccess)
        return fail(EVS_ERR_CUDA);
    if ((rc = dev_alloc(h->dev_allocs, &h->d_agg, cfg->max_batch))) return fail(rc);
    if ((rc = dev_alloc(h->dev_allocs, &h->d_idx[0], n_max))) return fail(rc);
    if ((rc = dev_alloc(h->dev_allocs, &h->d_out[0], n_max * cfg->dim))) return fail(rc);
    if ((rc = dev_alloc(h->dev_allocs, &h->d_hit[0], n_max))) return fail(rc);
    if ((rc = dev_alloc(h->dev_allocs, &P.flags, n_max))) return fail(rc);
    if ((rc = dev_alloc(h->dev_allocs, &P.pos_slot, n_max))) return fail(rc);
    if ((rc = dev_alloc(h->dev_allocs, &P.miss_list, n_max))) return fail(rc);
    if ((rc = dev_alloc(h->dev_allocs, &P.miss_ctl, 2))) return fail(rc);
    if ((rc = dev_alloc(h->dev_allocs, &P.hist, static_cast<size_t>(kSeqs) * n_chunks_max))) return fail(rc);
    if ((rc = dev_alloc(h->dev_allocs, &P.tot, kSeqs))) return fail(rc);
    if ((rc = dev_alloc(h->dev_allocs, &P.done, 1))) return fail(rc);
    if ((rc = dev_alloc(h->dev_allocs, &P.dbg, 32))) return fail(rc);

    if ((rc = build_tier(h, h->tier[0], cfg->main_precision, h->caps.c1, cfg->store_main))) return fail(rc);
    if (h->n_tiers == 2)
        if ((rc = build_tier(h, h->tier[1], cfg->secondary_precision, h->caps.c2, cfg->store_secondary))) return fail(rc);
    if (cfg->n_layers == 3 && h->caps.c3 > 0) {
        if ((rc = build_c3(h))) return fail(rc);
        h->c3_active = true;
    }
    P.tier[0] = h->tier[0].dev;
    if (h->n_tiers == 2) P.tier[1] = h->tier[1].dev;
    P.n_tiers = h->n_tiers;
    P.T = cfg->n_tables;
    P.D = cfg->dim;
    P.L = L;
    P.L_shift = L_shift;
    P.spc = spc;
    P.table_base = h->table_ids[0];
    for (int g = 0; g < kMaxTables; ++g) P.loc[g] = -1;
    for (int t = 0; t < cfg->n_tables; ++t) {
        P.tid[t] = h->table_ids[t];
        P.col[t] = t;                                   // evs_shard_connect switches to the global id
        P.loc[h->table_ids[t]] = t;
    }
    P.n_max = static_cast<unsigned>(n_max);
    {
        void *dp = nullptr;
        if (cudaHostGetDevicePointer(&dp, h->err_host, 0) != cudaSuccess) return fail(EVS_ERR_CUDA);
        P.err_host = static_cast<unsigned *>(dp);
        P.ring_host = reinterpret_cast<unsigned long long *>(static_cast<unsigned char *>(dp) + 64);
    }
    P.n_perfect_agg = h->cfg.n_tables_total;
    P.approx_thres = (h->n_tiers == 1) ? cfg->approx_emb_thres : 0;
    P.policy = cfg->policy;
    P.high_thres = h->cfg.high_agghit_threshold;
    P.n_chunks_max = n_chunks_max;
    {
        const char *qm = getenv("EVSTORE_B200_QUAD_MAX");          // tuning aid: largest serve grid whose k_update sums its predecessors directly
        P.quad_max = (qm && atoi(qm) > 0) ? atoi(qm) : kQuadMaxChunks;
        // CTAs of the miss-fetch role: ~512 64-byte row reads in flight (32 KB; fewer rows when they are larger) -- measured
        // optimum of profiles/r1_fetch_list_ab.md.  Rows that are 16-byte aligned are shared by groups of gsize lanes
        // (32 / gsize rows per warp and round), others take a whole warp each.
        {
            unsigned stride = h->tier[0].dev.row_stride;
            bool aligned = true;
            for (int i = 0; i < h->n_tiers; ++i) {
                stride = std::max(stride, h->tier[i].dev.row_stride);
                bool al = (h->tier[i].dev.row_bytes & 15u) == 0;
                for (const unsigned char *q : h->tier[i].store_dev) al = al && ((reinterpret_cast<uintptr_t>(q) & 15u) == 0);
                aligned = aligned && al;
            }
            int gsize = 32;
            if (aligned) {
                gsize = 1;
                while (gsize < static_cast<int>(stride >> 4) && gsize < 32) gsize <<= 1;
            }
            const int rows_per_cta = (kEvictThreads / 32) * (32 / gsize);
            // the link serves ~65 row reads / us whatever the row size up to 256 B once ~512-768 are in flight
            // (profiles/r2_zc_inflight.txt); the fetch role runs next to the eviction roles and keeps fewer
            // (r2: backing rows in evs_host_alloc memory take ~4x as many before the rate levels off, and the fetch role only
            // reads what the look-ahead did not stage)
            const bool big_pages = h->n_ranges > 0 && h->n_ranges_managed == h->n_ranges;
            const int target = big_pages ? static_cast<int>(std::min(2048u, std::max(512u, 131072u / stride)))
                                         : static_cast<int>(std::min(512u, std::max(256u, 65536u / stride)));
            h->fetch_list_ctas = std::max(1, (target + rows_per_cta - 1) / rows_per_cta);
            h->pf_ok = aligned;
            // the look-ahead kernel: nothing waits for it, so it keeps the link saturated (measured optimum for 64-byte
            // rows: 16 CTAs = 1024 rows; 8 or 12 leave rows unstaged, 32 slow k_update's atomics down)
            const int pf_target = big_pages ? (stride <= 64 ? 2048 : 1024) : (stride <= 64 ? 1024 : 768);
            h->pf_ctas = std::max(4, (pf_target + rows_per_cta - 1) / rows_per_cta);
        }
        const char *fc = getenv("EVSTORE_B200_FETCH_LIST_CTAS");   // tuning aid: CTAs of the fetch role = PCIe reads kept in flight
        if (fc && atoi(fc) > 0) h->fetch_list_ctas = atoi(fc);
        const char *pc = getenv("EVSTORE_B200_PF_CTAS");           // tuning aid: CTAs of k_prefetch
        if (pc && atoi(pc) > 0) h->pf_ctas = atoi(pc);
        const char *pm = getenv("EVSTORE_B200_PF_MODE");           // experiments: 1 = probe + L2 warm-up only (no staging)
        h->pf_mode = (pm && pm[0] == '1') ? 1 : 0;
        const char *pw = getenv("EVSTORE_B200_PF_WAIT");           // experiments: 1 = stream-event wait for the staging buffer as well
        h->pf_wait_mode = (pw && pw[0] == '1') ? 1 : 0;
        const char *pe = getenv("EVSTORE_B200_NO_PREFETCH");       // tuning aid: evs_prefetch becomes a no-op
        if (pe && pe[0] == '1') h->pf_ok = false;
        // CTAs of k_evict per tier = 256-record chunks of the rings examined at once.  A batch evicts about as many keys
        // as it misses (a few per cent of its positions) and most records at the ring heads are live, so one chunk per
        // 2048 positions covers the usual batch several times over (configs[1]: victims complete after 5-7 chunks of 26);
        // batches that need more take further chunks by ticket.  More CTAs only add DRAM reads (ncu: 8.3 MB -> 1.2 MB).
        h->evict_ctas = static_cast<int>(std::min<long long>(kTierCtas, std::max<long long>(16, n_max / 2048)));
        const char *ec = getenv("EVSTORE_B200_EVICT_CTAS");        // tuning aid (<= 256)
        if (ec && atoi(ec) > 0) h->evict_ctas = std::min(atoi(ec), kEvictThreads);
        const char *pd = getenv("EVSTORE_B200_PDL");               // tuning aid: 0 = plain stream order between the batch's kernels
        h->use_pdl = !(pd && pd[0] == '0');
    }
    P.evict_ctas = h->evict_ctas;
    P.fetch_ctas = h->fetch_list_ctas;
    P.pdl = h->use_pdl ? 1 : 0;
    P.rows = h->d_rows;
    P.args = h->d_args;
    P.g = h->g;
    for (int i = 0; i < h->n_tiers; ++i) {
        bool al = (h->tier[i].dev.row_bytes & 15u) == 0;
        for (const unsigned char *q : h->tier[i].store_dev) al = al && ((reinterpret_cast<uintptr_t>(q) & 15u) == 0);
        if (al) P.store_aligned |= 1 << i;
    }
    P.stage_stride = std::max(h->tier[0].dev.row_stride, h->n_tiers == 2 ? h->tier[1].dev.row_stride : 0u);
    const size_t us = fetch_smem(h);
    if (us > 32 * 1024) {
        const KernelSet ks = kernels_of_handle(h);
        if (cudaFuncSetAttribute(reinterpret_cast<const void *>(ks.evict), cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 static_cast<int>(us)) != cudaSuccess) {
            set_error("row too large for the fetch role's staging buffer");
            return fail(EVS_ERR_INVALID);
        }
    }
    if (h->pf_ok) {
        // staging rows of the look-ahead: two parities, one row_stride slot per position
        if ((rc = dev_alloc(h->dev_allocs, &P.pf_tag, 2 * static_cast<size_t>(n_max)))) return fail(rc);
        if ((rc = dev_alloc(h->dev_allocs, &P.pf_rows, 2 * static_cast<size_t>(n_max) * P.stage_stride, false))) return fail(rc);
    }
    const char *ng = getenv("EVSTORE_B200_NO_GRAPH");
    h->use_graph = !(ng && ng[0] == '1');
    if (h->use_graph && (rc = build_graph(h))) {
        if (!h->use_pdl) return fail(rc);
        // a driver that cannot capture programmatic edges: plain stream order between the kernels
        fprintf(stderr, "evstore_b200: graph capture with programmatic dependent launch failed (%s); retrying without\n", evs_last_error());
        cudaGetLastError();
        h->use_pdl = false;
        P.pdl = 0;
        destroy_graphs(h);
        if ((rc = build_graph(h))) return fail(rc);
    }
    *out = h;
    return EVS_OK;
}

int evs_destroy(evs_handle h) {
    if (h == nullptr) return EVS_ERR_INVALID;
    free_all(h);
    return EVS_OK;
}

static int set_serve_params(evs_handle h, cudaGraphExec_t exec, cudaGraphNode_t node, BatchArgs &a) {
    const KernelSet ks = kernels_of_handle(h);
    void *kargs[] = {&h->params, &a};
    cudaKernelNodeParams kp{};
    kp.func = reinterpret_cast<void *>(serve_of(h, ks));
    kp.gridDim = dim3(h->params.n_chunks_max);
    kp.blockDim = dim3(kLookupThreads);
    kp.sharedMemBytes = 0;
    kp.kernelParams = kargs;
    EVS_CUDA(cudaGraphExecKernelNodeSetParams(exec, node, &kp));
    return EVS_OK;
}

static void count_batch_launches(evs_handle h) {
    h->prof.launches[K_SERVE]++, h->prof.launches[K_UPDATE]++, h->prof.launches[K_EVICT]++;
    if (h->params.n_chunks_max > h->params.quad_max) h->prof.launches[K_SCAN]++;
}

// CTAs of k_serve / k_update for B samples.
static int serve_ctas(evs_handle h, int32_t B) { return (B + h->params.spc - 1) / h->params.spc; }

// The stream a call is ordered on: the caller's, else the handle's own.
static cudaStream_t stream_of(evs_handle h, void *stream) { return stream ? static_cast<cudaStream_t>(stream) : h->stream; }

// The arguments of a lookup of B samples; out_stride <= 0: rows packed as [B][n_tables][dim].
static BatchArgs lookup_args(evs_handle h, const int64_t *idx, int32_t B, float *out, int64_t out_stride, uint8_t *hit) {
    BatchArgs a{};
    a.idx = reinterpret_cast<const long long *>(idx);
    a.B = B;
    a.out = out;
    a.out_stride = out_stride > 0 ? out_stride : static_cast<long long>(h->cfg.n_tables) * h->cfg.dim;
    a.hit = hit;
    a.agg_out = h->d_agg;
    return a;
}

// Launch k_prefetch for batch number `seq` with generation `gen` on the look-ahead stream.  The kernel itself waits (on the
// device) until the staging rows of its parity are free, i.e. until the miss-fetch role of batch seq - 2 has finished.
static int launch_prefetch(evs_handle h, const int64_t *idx_dev, int32_t B, uint64_t seq, uint32_t gen) {
    PrefetchArgs pa{};
    pa.idx = reinterpret_cast<const long long *>(idx_dev);
    pa.B = B;
    pa.seq = static_cast<unsigned>(seq);
    pa.gen = gen;
    pa.mode = h->pf_mode;
    const KernelSet ks = kernels_of_handle(h);
    const int S = pf_tile_samples(h->cfg.n_tables);
    const int n_tiles = (B + S - 1) / S;
    LaunchScope ls(h->prof, K_PREFETCH, h->pf_stream);
    void *args[] = {&h->params, &pa};
    EVS_CUDA(launch_ex(reinterpret_cast<const void *>(ks.prefetch), dim3(std::min(h->pf_ctas, n_tiles)), kPfThreads, 0, h->pf_stream,
                       args, false));
    return EVS_OK;
}

// The next announcement's generation (tags are generation << 1 | tier: start over with clean tags before they wrap).
static int next_pf_gen(evs_handle h, uint32_t *gen) {
    if (++h->pf.gen >= 0x7FFFFFFFu) {
        EVS_CUDA(cudaStreamSynchronize(h->stream));
        EVS_CUDA(cudaMemsetAsync(h->params.pf_tag, 0, 2 * sizeof(unsigned) * static_cast<size_t>(h->params.n_max), h->pf_stream));
        h->pf.gen = 1;
    }
    *gen = h->pf.gen;
    return EVS_OK;
}

// Look-ahead for the next batch (see evs_prefetch.cuh).  ready: event after which idx_dev is complete, or null.
static int prefetch_next(evs_handle h, const int64_t *idx_dev, int32_t B, cudaEvent_t ready) {
    if (!h->pf_ok) return EVS_OK;
    const uint64_t seq = h->seq + 1;
    if (h->pf.matches(seq, idx_dev, B)) return EVS_OK;   // already announced
    if (ready) EVS_CUDA(cudaStreamWaitEvent(h->pf_stream, ready, 0));
    if (h->pf_wait_mode == 1 && h->ev_done_valid[seq & 1]) EVS_CUDA(cudaStreamWaitEvent(h->pf_stream, h->ev_done[seq & 1], 0));
    uint32_t gen = 0;
    int rc = next_pf_gen(h, &gen);
    if (rc) return rc;
    if ((rc = launch_prefetch(h, idx_dev, B, seq, gen))) return rc;
    h->pf.record(seq, idx_dev, B);
    return EVS_OK;
}

// A probe pass (evs_probe_batch, and the first pass of a sharded batch without the one-pass exchange): k_serve counts
// every sample's hits and returns.  It is not a batch: no batch number, no bookkeeping, no ring appends.
static int launch_probe(evs_handle h, BatchArgs a, cudaStream_t st) {
    a.probe_only = 1;
    LaunchScope ls(h->prof, K_PROBE, st);
    EVS_CUDA(launch_serve(serve_of(h, kernels_of_handle(h)), serve_ctas(h, a.B), st, h->params, a));
    return EVS_OK;
}

// Submit a call's n consecutive batches of B samples on st: the one place that numbers batches, matches them with the
// look-ahead and keeps the books.  fill(i, a) sets the arguments of batch i (a.idx = idx[i]) just before the batch is
// submitted, in order; it may enqueue work on st ahead of the batch, and returns an error code.  may_group: the caller
// allows h->group batches in one graph launch.
extern "C++" {                                           // a template cannot have C linkage
template <class Fill>
static int submit_batches(evs_handle h, cudaStream_t st, int n, const int64_t *const *idx, int32_t B, bool may_group, Fill &&fill) {
    // The caller is capturing its own graph (e.g. a whole sequential_forward): the batches go in as plain kernels with
    // frozen arguments; the device numbers each replay itself (BatchArgs::seq == 0, pf_gen == 0) and the host is told by
    // evs_note_replays.
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(st, &cs) == cudaSuccess && cs == cudaStreamCaptureStatusActive) {
        for (int i = 0; i < n; ++i) {
            BatchArgs a{};
            int rc = fill(i, a);
            if (rc || (rc = enqueue_batch(h, st, serve_ctas(h, a.B), a, false))) return rc;
        }
        return EVS_OK;
    }
    const int G = h->group;
    for (int i = 0; i < n;) {
        // A group is one graph launch: the batches stay strictly ordered -- the graph is the same linear chain of kernels --
        // but only the first k_serve pays a graph-to-graph boundary; the others follow their predecessor's k_evict over a
        // programmatic edge.  Every bucket ring must take the whole group's appends (the host tracks an upper bound of the
        // occupancy).
        bool grouped = may_group && h->use_graph && !h->prof.on && G > 1 && h->ggraph != nullptr && h->pf_wait_mode == 0 && n - i >= G;
        for (int t = 0; t < h->n_tiers && grouped; ++t) {
            int rc = maintain_rings(h, t, st, G + 1);
            if (rc) return rc;
            grouped = ring_fits(h, t, G + 1);
        }
        const int m = grouped ? G : 1;
        const uint64_t seq0 = h->seq + 1;
        BatchArgs a[evs_handle_s::kGroup];
        uint32_t gens[evs_handle_s::kGroup] = {};
        for (int k = 0; k < m; ++k) {
            a[k] = BatchArgs{};
            int rc = fill(i + k, a[k]);
            if (rc) return rc;
            a[k].seq = static_cast<unsigned>(seq0 + k);
            // rows staged by evs_prefetch are used when the announcement matches the batch; the later batches of a group
            // are announced here, and their k_prefetch follows the graph launch
            if (k == 0) {
                a[k].pf_gen = h->pf.matches(seq0, a[k].idx, a[k].B) ? h->pf.gen : 0u;
            } else if (h->pf_ok) {
                if ((rc = next_pf_gen(h, &gens[k]))) return rc;
                a[k].pf_gen = gens[k];
            }
        }
        if (h->use_graph && !h->prof.on) {
            const cudaGraphExec_t exec = grouped ? h->ggraph : h->graph;
            for (int k = 0; k < m; ++k) {
                int rc = set_serve_params(h, exec, grouped ? h->gserve[k] : h->serve_node, a[k]);
                if (rc) return rc;
            }
            EVS_CUDA(cudaGraphLaunch(exec, st));
            for (int k = 0; k < m; ++k) count_batch_launches(h);
        } else {
            // outside a graph the chain continues across batches: k_serve is a programmatic dependent of whatever kernel
            // precedes it on the stream (the previous batch's k_evict in a serving loop)
            int rc = enqueue_batch(h, st, serve_ctas(h, a[0].B), a[0], true);
            if (rc) return rc;
        }
        h->seq += m;
        h->batches += m;
        if (grouped) {
            if (h->pf_ok) {
                for (int k = 1; k < m; ++k) {
                    int rc = launch_prefetch(h, reinterpret_cast<const int64_t *>(a[k].idx), a[k].B, seq0 + k, gens[k]);
                    if (rc) return rc;
                }
                h->pf.record(seq0 + m - 1, a[m - 1].idx, a[m - 1].B);
            }
        } else {
            // the staging rows of this parity may be overwritten (by the look-ahead for batch seq + 2) once this batch is done
            if (h->pf_wait_mode == 1) {
                EVS_CUDA(cudaEventRecord(h->ev_done[seq0 & 1], st));
                h->ev_done_valid[seq0 & 1] = true;
            }
            for (int t = 0; t < h->n_tiers; ++t) {
                int rc = maintain_rings(h, t, st);
                if (rc) return rc;
            }
            // the batch after it is announced so that its misses are staged as inside a group
            if (i + 1 < n) {
                int rc = prefetch_next(h, idx[i + 1], B, nullptr);
                if (rc) return rc;
            }
        }
        i += m;
    }
    return EVS_OK;
}
}  // extern "C++"

// One batch whose arguments the caller built.
static int submit_batch(evs_handle h, cudaStream_t st, const BatchArgs &a) {
    const int64_t *idx = reinterpret_cast<const int64_t *>(a.idx);
    return submit_batches(h, st, 1, &idx, a.B, false, [&](int, BatchArgs &b) {
        b = a;
        return EVS_OK;
    });
}

int evs_prefetch(evs_handle h, const int64_t *idx_dev, int32_t B, void *ready_event) {
    if (h == nullptr || idx_dev == nullptr || B < 1 || B > h->cfg.max_batch) {
        set_error("evs_prefetch: bad handle / B / pointer");
        return EVS_ERR_INVALID;
    }
    DeviceGuard dg(h->cfg.device);
    return prefetch_next(h, idx_dev, B, static_cast<cudaEvent_t>(ready_event));
}

int evs_lookup_batch(evs_handle h, const int64_t *idx_dev, int32_t B, float *out_dev, int64_t out_stride,
                     uint8_t *hit_dev, const uint8_t *agg_in, void *stream) {
    if (h == nullptr || B < 0 || B > h->cfg.max_batch || (B > 0 && (idx_dev == nullptr || out_dev == nullptr))) {
        set_error("evs_lookup_batch: bad handle / B / pointers");
        return EVS_ERR_INVALID;
    }
    if (B == 0) return EVS_OK;
    DeviceGuard dg(h->cfg.device);
    BatchArgs a = lookup_args(h, idx_dev, B, out_dev, out_stride, hit_dev);
    a.agg_in = agg_in;
    return submit_batch(h, stream_of(h, stream), a);
}

int evs_lookup_batches(evs_handle h, int32_t n, const int64_t *const *idx_dev, int32_t B, float *const *out_dev, int64_t out_stride,
                       uint8_t *const *hit_dev, void *stream) {
    if (h == nullptr || n < 0 || B < 1 || B > h->cfg.max_batch || (n > 0 && (idx_dev == nullptr || out_dev == nullptr))) {
        set_error("evs_lookup_batches: bad handle / n / B / pointers");
        return EVS_ERR_INVALID;
    }
    for (int i = 0; i < n; ++i)
        if (idx_dev[i] == nullptr || out_dev[i] == nullptr) {
            set_error("evs_lookup_batches: null batch pointer");
            return EVS_ERR_INVALID;
        }
    DeviceGuard dg(h->cfg.device);
    return submit_batches(h, stream_of(h, stream), n, idx_dev, B, !h->sharded, [&](int i, BatchArgs &a) {
        a = lookup_args(h, idx_dev[i], B, out_dev[i], out_stride, hit_dev ? hit_dev[i] : nullptr);
        return EVS_OK;
    });
}

// Bags (pooling factor > 1) on the cached path: see evs_bags.cuh.
static int bags_check(evs_handle h, const char *what, const int64_t *idx_dev, const int64_t *off_dev, int32_t B, int64_t nnz,
                      int32_t max_per_bag, long long max_slices) {
    if (h == nullptr || B < 0 || nnz < 0 || max_per_bag < 1 || max_per_bag > kMaxPerBag || off_dev == nullptr ||
        (nnz > 0 && idx_dev == nullptr)) {
        set_error(std::string(what) + ": bad handle / B / nnz / max_per_bag (1..32) / pointers");
        return EVS_ERR_INVALID;
    }
    if (static_cast<long long>(B) * max_per_bag > max_slices) {
        set_error(std::string(what) + ": B * max_per_bag slices exceed the largest batch (max_batch, or batch_max of evs_shard_create)");
        return EVS_ERR_INVALID;
    }
    return EVS_OK;
}

// The batch's slices: scratch on first use (slice rows W tables wide: a table's rows sit at its output column p.col[t],
// which is its global id once the handle is a rank of a sharded cache), then k_bags_expand.
static int bags_expand(evs_handle h, cudaStream_t st, const int64_t *idx_dev, const int64_t *off_dev, int32_t B, int64_t nnz, int P) {
    const int T = h->cfg.n_tables, D = h->cfg.dim;
    const int W = h->sharded ? h->cfg.n_tables_total : T;
    if (h->bag_idx == nullptr || h->bag_cols < W) {
        t_alloc_bytes = &h->hbm_bytes;
        struct AllocScope {
            ~AllocScope() { t_alloc_bytes = nullptr; }
        } alloc_scope;
        const long long n_max = static_cast<long long>(h->cfg.max_batch) * T;
        int rc;
        if (h->bag_idx == nullptr) {
            if ((rc = dev_alloc(h->dev_allocs, &h->bag_idx, n_max))) return rc;
            if ((rc = dev_alloc(h->dev_allocs, &h->bag_hit, n_max))) return rc;
        } else {                                              // bags before evs_shard_connect: the rows grow to W tables
            EVS_CUDA(cudaDeviceSynchronize());
            h->dev_allocs.erase(std::find(h->dev_allocs.begin(), h->dev_allocs.end(), static_cast<void *>(h->bag_rows)));
            EVS_CUDA(cudaFree(h->bag_rows));
            h->hbm_bytes -= static_cast<size_t>(h->cfg.max_batch) * h->bag_cols * D * sizeof(float);
        }
        if ((rc = dev_alloc(h->dev_allocs, &h->bag_rows, static_cast<long long>(h->cfg.max_batch) * W * D))) return rc;
        h->bag_cols = W;
    }
    const long long total = static_cast<long long>(B) * P * T;
    LaunchScope ls(h->prof, K_BAGS, st);
    k_bags_expand<<<static_cast<unsigned>(std::min<long long>((total + 255) / 256, 148 * 8)), 256, 0, st>>>(
        h->params, reinterpret_cast<const long long *>(idx_dev), reinterpret_cast<const long long *>(off_dev), B, P, nnz, h->bag_idx);
    EVS_CUDA(cudaGetLastError());
    return EVS_OK;
}

// The arguments of the slice batch bags_expand staged: B*P slices, rows into the slice staging.
static BatchArgs bags_args(evs_handle h, int32_t B, int P) {
    BatchArgs a = lookup_args(h, reinterpret_cast<const int64_t *>(h->bag_idx), B * P, h->bag_rows,
                              static_cast<long long>(h->bag_cols) * h->cfg.dim, h->bag_hit);
    a.bags = 1;
    return a;
}

// k_bags_pool over the staged slice rows: into out (one GPU) or, sh.world > 1, into the owner ranks' receive buffers.
static int bags_pool(evs_handle h, cudaStream_t st, const ShardArgs &sh, const int64_t *off_dev, int32_t B, int P, int64_t nnz, float *out_dev,
                     int64_t out_stride, uint8_t *hit_dev) {
    LaunchScope ls(h->prof, K_BAGS, st);
    const int T = h->cfg.n_tables, D = h->cfg.dim;
    const long long os = out_stride > 0 ? out_stride : static_cast<long long>(T) * D;
    const bool vec = (D & 3) == 0 && (sh.world > 1 || ((os & 3) == 0 && (reinterpret_cast<uintptr_t>(out_dev) & 15u) == 0));
    const long long items = static_cast<long long>(B) * T * (vec ? D / 4 : D);
    const unsigned grid = static_cast<unsigned>(std::min<long long>((items + 255) / 256, 148 * 16));
    const long long *off = reinterpret_cast<const long long *>(off_dev);
    if (vec)
        k_bags_pool<true><<<grid, 256, 0, st>>>(h->params, sh, h->bag_rows, h->bag_hit, off, B, P, nnz, h->bag_cols, out_dev, os, hit_dev);
    else
        k_bags_pool<false><<<grid, 256, 0, st>>>(h->params, sh, h->bag_rows, h->bag_hit, off, B, P, nnz, h->bag_cols, out_dev, os, hit_dev);
    EVS_CUDA(cudaGetLastError());
    return EVS_OK;
}

static int lookup_bags(evs_handle h, const char *what, const int64_t *idx_dev, const int64_t *off_dev, int32_t B, int64_t nnz,
                       int32_t max_per_bag, float *out_dev, int64_t out_stride, uint8_t *hit_dev, const uint8_t *agg_in, void *stream) {
    int rc = bags_check(h, what, idx_dev, off_dev, B, nnz, max_per_bag, h ? h->cfg.max_batch : 0);
    if (rc) return rc;
    if (B > 0 && out_dev == nullptr) {
        set_error(std::string(what) + ": null output");
        return EVS_ERR_INVALID;
    }
    if (h->sharded) {
        set_error(std::string(what) + ": not available on a rank of a table-wise sharded cache (evs_shard_lookup_bags is)");
        return EVS_ERR_INVALID;
    }
    if (B == 0) return EVS_OK;
    DeviceGuard dg(h->cfg.device);
    cudaStream_t st = stream_of(h, stream);
    const int P = max_per_bag;
    if ((rc = bags_expand(h, st, idx_dev, off_dev, B, nnz, P))) return rc;
    BatchArgs a = bags_args(h, B, P);
    a.agg_in = agg_in;
    if ((rc = submit_batch(h, st, a))) return rc;
    return bags_pool(h, st, ShardArgs{}, off_dev, B, P, nnz, out_dev, out_stride, hit_dev);
}

int evs_lookup_bags(evs_handle h, const int64_t *idx_dev, const int64_t *off_dev, int32_t B, int64_t nnz, int32_t max_per_bag,
                    float *out_dev, int64_t out_stride, uint8_t *hit_dev, void *stream) {
    return lookup_bags(h, "evs_lookup_bags", idx_dev, off_dev, B, nnz, max_per_bag, out_dev, out_stride, hit_dev, nullptr, stream);
}

int evs_lookup_bags_agg(evs_handle h, const int64_t *idx_dev, const int64_t *off_dev, int32_t B, int64_t nnz, int32_t max_per_bag,
                        float *out_dev, int64_t out_stride, uint8_t *hit_dev, const uint8_t *agg_in, void *stream) {
    if (agg_in == nullptr && B > 0) {
        set_error("evs_lookup_bags_agg: null agg_in");
        return EVS_ERR_INVALID;
    }
    return lookup_bags(h, "evs_lookup_bags_agg", idx_dev, off_dev, B, nnz, max_per_bag, out_dev, out_stride, hit_dev, agg_in, stream);
}

int evs_probe_bags(evs_handle h, const int64_t *idx_dev, const int64_t *off_dev, int32_t B, int64_t nnz, int32_t max_per_bag,
                   uint8_t *agg_out_dev, void *stream) {
    int rc = bags_check(h, "evs_probe_bags", idx_dev, off_dev, B, nnz, max_per_bag, h ? h->cfg.max_batch : 0);
    if (rc) return rc;
    if (B > 0 && agg_out_dev == nullptr) {
        set_error("evs_probe_bags: null agg_out");
        return EVS_ERR_INVALID;
    }
    if (B == 0) return EVS_OK;
    DeviceGuard dg(h->cfg.device);
    cudaStream_t st = stream_of(h, stream);
    if ((rc = bags_expand(h, st, idx_dev, off_dev, B, nnz, max_per_bag))) return rc;
    BatchArgs a = bags_args(h, B, max_per_bag);
    a.agg_out = agg_out_dev;
    return launch_probe(h, a, st);
}

// New values for the rows of n keys (evs_refresh.cuh), stream-ordered between batches.
int evs_update_rows(evs_handle h, const int64_t *keys_dev, int64_t n, const float *values_dev, int64_t value_stride,
                    uint8_t *where_dev, void *stream) {
    if (h == nullptr || n < 0 || value_stride < 0 || (value_stride > 0 && value_stride < h->cfg.dim) ||
        (n > 0 && (keys_dev == nullptr || values_dev == nullptr))) {
        set_error("evs_update_rows: bad handle / n / value_stride (0 or >= dim) / pointers");
        return EVS_ERR_INVALID;
    }
    if (n == 0) return EVS_OK;
    DeviceGuard dg(h->cfg.device);
    cudaStream_t st = stream_of(h, stream);
    {
        cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
        if (cudaStreamIsCapturing(st, &cs) == cudaSuccess && cs != cudaStreamCaptureStatusNone) {
            set_error("evs_update_rows: the stream is being captured; call it outside a graph, between launches");
            return EVS_ERR_INVALID;
        }
    }
    const RefreshFn fn = kernels_of_handle(h).update_rows;
    if (fn == nullptr) return EVS_ERR_INVALID;
    if (n > (1ll << 30)) {
        set_error("evs_update_rows: at most 2^30 keys per call");
        return EVS_ERR_INVALID;
    }
    // scratch hash at a load factor <= 1/2; a larger call grows it synchronously (the previous call may still read it)
    const size_t cap = next_pow2(static_cast<unsigned long long>(std::max<int64_t>(2 * n, 1024)));
    if (cap > h->upd_cap) {
        EVS_CUDA(cudaDeviceSynchronize());
        if (h->upd_key) cudaFree(h->upd_key);
        if (h->upd_pos) cudaFree(h->upd_pos);
        h->upd_key = nullptr;
        h->upd_pos = nullptr;
        h->hbm_bytes -= h->upd_cap * (sizeof(unsigned long long) + sizeof(long long));
        h->upd_cap = 0;
        EVS_CUDA(cudaMalloc(&h->upd_key, cap * sizeof(unsigned long long)));
        EVS_CUDA(cudaMalloc(&h->upd_pos, cap * sizeof(long long)));
        h->upd_cap = cap;
        h->hbm_bytes += cap * (sizeof(unsigned long long) + sizeof(long long));
    }
    if (h->ev_upd == nullptr) EVS_CUDA(cudaEventCreateWithFlags(&h->ev_upd, cudaEventDisableTiming));
    RefreshArgs ra{};
    ra.keys = reinterpret_cast<const long long *>(keys_dev);
    ra.n = n;
    ra.values = values_dev;
    ra.vstride = value_stride > 0 ? value_stride : h->cfg.dim;
    ra.where = where_dev;
    ra.hkey = h->upd_key;
    ra.hpos = h->upd_pos;
    ra.hmask = static_cast<unsigned>(cap - 1);
    ra.gsize = 1;
    while (ra.gsize < 32 && 8 * ra.gsize < h->cfg.dim) ra.gsize <<= 1;
    EVS_CUDA(cudaMemsetAsync(h->upd_key, 0xFF, cap * sizeof(unsigned long long), st));
    EVS_CUDA(cudaMemsetAsync(h->upd_pos, 0xFF, cap * sizeof(long long), st));
    void *args[] = {&h->params, &ra};
    const long long per_cta = static_cast<long long>(kRefreshThreads / 32) * (32 / ra.gsize);
    {
        LaunchScope ls(h->prof, K_UPDATE_ROWS, st);
        const unsigned g1 = static_cast<unsigned>(std::min<long long>((n + kRefreshThreads - 1) / kRefreshThreads, 148 * 16));
        EVS_CUDA(launch_ex(reinterpret_cast<const void *>(k_update_rows_claim), dim3(g1), kRefreshThreads, 0, st, args, false));
        // no programmatic serialization, here or in the claim: the next batch's k_serve (a programmatic dependent of
        // whatever precedes it) cannot start before every row is written
        const unsigned g2 = static_cast<unsigned>(std::min<long long>((n + per_cta - 1) / per_cta, 148 * 16));
        EVS_CUDA(launch_ex(reinterpret_cast<const void *>(fn), dim3(g2), kRefreshThreads, 0, st, args, false));
    }
    // The look-ahead: an announcement made before this call may have staged old bytes (or may still be staging them).
    // Cancel it -- the next batch fetches its misses itself; a k_prefetch still running tags its rows with a generation
    // no later batch asks for -- and order every later k_prefetch behind the new bytes.
    h->pf.cancel();
    EVS_CUDA(cudaEventRecord(h->ev_upd, st));
    EVS_CUDA(cudaStreamWaitEvent(h->pf_stream, h->ev_upd, 0));
    return EVS_OK;
}

int evs_note_replays(evs_handle h, int64_t n, void *stream) {
    if (h == nullptr || n < 0) return EVS_ERR_INVALID;
    DeviceGuard dg(h->cfg.device);
    cudaStream_t st = stream_of(h, stream);
    h->seq += static_cast<uint64_t>(n);
    h->batches += static_cast<uint64_t>(n);
    for (int i = 0; i < h->n_tiers; ++i) {
        int rc = maintain_rings(h, i, st);
        if (rc) return rc;
    }
    return poll_error(h);
}

int evs_probe_batch(evs_handle h, const int64_t *idx_dev, int32_t B, uint8_t *agg_out_dev, void *stream) {
    if (h == nullptr || B < 0 || B > h->cfg.max_batch || idx_dev == nullptr || agg_out_dev == nullptr) return EVS_ERR_INVALID;
    if (B == 0) return EVS_OK;
    DeviceGuard dg(h->cfg.device);
    BatchArgs a{};
    a.idx = reinterpret_cast<const long long *>(idx_dev);
    a.agg_out = agg_out_dev;
    a.B = B;
    return launch_probe(h, a, stream_of(h, stream));
}

// The device error word as the host sees it (the kernels mirror it into pinned memory): sticky until cleared.
static int poll_error(evs_handle h) {
    const unsigned e = *reinterpret_cast<volatile unsigned *>(h->err_host);
    if (e != 0u && h->sticky_error == 0) h->sticky_error = (e == 7u) ? EVS_ERR_PEER : EVS_ERR_INDEX;
    if (h->sticky_error == EVS_ERR_PEER) set_error("a peer rank did not deliver its hit counts / rows in time (table-wise sharding)");
    else if (h->sticky_error == EVS_ERR_INDEX) set_error("an index was outside [0, rows[table]); the lookup was answered from row 0");
    return h->sticky_error;
}

int evs_check(evs_handle h, int clear) {
    if (h == nullptr) return EVS_ERR_INVALID;
    const int rc = poll_error(h);
    if (clear) {
        h->sticky_error = 0;
        *reinterpret_cast<volatile unsigned *>(h->err_host) = 0u;
    }
    return rc;
}

int evs_memory_footprint(evs_handle h, uint64_t *hbm_bytes) {
    if (h == nullptr || hbm_bytes == nullptr) return EVS_ERR_INVALID;
    *hbm_bytes = h->hbm_bytes;
    return EVS_OK;
}

int evs_lookup_batch_host(evs_handle h, const int64_t *idx_host, int32_t B, float *out_host, uint8_t *hit_host) {
    if (h == nullptr || B < 0 || B > h->cfg.max_batch || (B > 0 && (idx_host == nullptr || out_host == nullptr))) {
        set_error("evs_lookup_batch_host: bad handle / B / pointers");
        return EVS_ERR_INVALID;
    }
    if (B == 0) return EVS_OK;
    DeviceGuard dg(h->cfg.device);
    // staging slot 0 is shared with the pipelined path: wait for a ticket that may still be copying out of it
    if (h->s_out != nullptr) EVS_CUDA(cudaStreamSynchronize(h->s_out));
    const size_t n = static_cast<size_t>(B) * h->cfg.n_tables;
    EVS_CUDA(cudaMemcpyAsync(h->d_idx[0], idx_host, n * sizeof(int64_t), cudaMemcpyHostToDevice, h->stream));
    int rc = evs_lookup_batch(h, reinterpret_cast<const int64_t *>(h->d_idx[0]), B, h->d_out[0], 0, h->d_hit[0], nullptr, h->stream);
    if (rc) return rc;
    EVS_CUDA(cudaMemcpyAsync(out_host, h->d_out[0], n * h->cfg.dim * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    if (hit_host != nullptr) EVS_CUDA(cudaMemcpyAsync(hit_host, h->d_hit[0], n, cudaMemcpyDeviceToHost, h->stream));
    EVS_CUDA(cudaStreamSynchronize(h->stream));
    return poll_error(h);
}

// Pipelined host-buffer path.  evs_submit_host returns at once with a ticket; at most kPipeSlots
// batches are in flight (the call blocks on the oldest one when all slots are taken).  The copies
// run on their own streams, so the H2D of batch n+1 and the D2H of batch n-1 overlap the kernels
// of batch n; the batches themselves stay strictly ordered.
static int pipe_init(evs_handle h) {
    if (h->s_in != nullptr) return EVS_OK;
    t_alloc_bytes = &h->hbm_bytes;
    struct AllocScope {
        ~AllocScope() { t_alloc_bytes = nullptr; }
    } alloc_scope;
    const long long n_max = static_cast<long long>(h->cfg.max_batch) * h->cfg.n_tables;
    EVS_CUDA(cudaStreamCreateWithFlags(&h->s_in, cudaStreamNonBlocking));
    EVS_CUDA(cudaStreamCreateWithFlags(&h->s_out, cudaStreamNonBlocking));
    int rc;
    for (int i = 0; i < evs_handle_s::kPipeSlots; ++i) {
        if (i > 0) {
            if ((rc = dev_alloc(h->dev_allocs, &h->d_idx[i], n_max))) return rc;
            if ((rc = dev_alloc(h->dev_allocs, &h->d_out[i], n_max * h->cfg.dim))) return rc;
            if ((rc = dev_alloc(h->dev_allocs, &h->d_hit[i], n_max))) return rc;
        }
        EVS_CUDA(cudaEventCreateWithFlags(&h->ev_in[i], cudaEventDisableTiming));
        EVS_CUDA(cudaEventCreateWithFlags(&h->ev_comp[i], cudaEventDisableTiming));
        EVS_CUDA(cudaEventCreateWithFlags(&h->ev_out[i], cudaEventDisableTiming));
    }
    return EVS_OK;
}

int evs_submit_host(evs_handle h, const int64_t *idx_host, int32_t B, float *out_host, uint8_t *hit_host, int64_t *ticket) {
    if (h == nullptr || B < 1 || B > h->cfg.max_batch || idx_host == nullptr || out_host == nullptr) {
        set_error("evs_submit_host: bad handle / B / pointers");
        return EVS_ERR_INVALID;
    }
    DeviceGuard dg(h->cfg.device);
    int rc = pipe_init(h);
    if (rc) return rc;
    const int slot = static_cast<int>(h->submitted % evs_handle_s::kPipeSlots);
    if (h->submitted >= evs_handle_s::kPipeSlots) EVS_CUDA(cudaEventSynchronize(h->ev_out[slot]));   // slot free again
    const size_t n = static_cast<size_t>(B) * h->cfg.n_tables;
    EVS_CUDA(cudaMemcpyAsync(h->d_idx[slot], idx_host, n * sizeof(int64_t), cudaMemcpyHostToDevice, h->s_in));
    EVS_CUDA(cudaEventRecord(h->ev_in[slot], h->s_in));
    // look-ahead: the indices are on the device long before the batches queued ahead of this one have run
    if ((rc = prefetch_next(h, reinterpret_cast<const int64_t *>(h->d_idx[slot]), B, h->ev_in[slot]))) return rc;
    EVS_CUDA(cudaStreamWaitEvent(h->stream, h->ev_in[slot], 0));
    rc = evs_lookup_batch(h, reinterpret_cast<const int64_t *>(h->d_idx[slot]), B, h->d_out[slot], 0, h->d_hit[slot], nullptr,
                          h->stream);
    if (rc) return rc;
    EVS_CUDA(cudaEventRecord(h->ev_comp[slot], h->stream));
    EVS_CUDA(cudaStreamWaitEvent(h->s_out, h->ev_comp[slot], 0));
    EVS_CUDA(cudaMemcpyAsync(out_host, h->d_out[slot], n * h->cfg.dim * sizeof(float), cudaMemcpyDeviceToHost, h->s_out));
    if (hit_host != nullptr) EVS_CUDA(cudaMemcpyAsync(hit_host, h->d_hit[slot], n, cudaMemcpyDeviceToHost, h->s_out));
    EVS_CUDA(cudaEventRecord(h->ev_out[slot], h->s_out));
    if (ticket) *ticket = h->submitted;
    h->submitted++;
    return EVS_OK;
}

int evs_wait_host(evs_handle h, int64_t ticket) {
    if (h == nullptr || ticket < 0 || ticket >= h->submitted) return EVS_ERR_INVALID;
    if (ticket + evs_handle_s::kPipeSlots < h->submitted) return poll_error(h);   // its slot was already recycled => done
    EVS_CUDA(cudaEventSynchronize(h->ev_out[ticket % evs_handle_s::kPipeSlots]));
    return poll_error(h);
}

int evs_sync(evs_handle h) {
    if (h == nullptr) return EVS_ERR_INVALID;
    EVS_CUDA(cudaSetDevice(h->cfg.device));
    EVS_CUDA(cudaDeviceSynchronize());
    return check_device_errors(h);
}

int evs_stats(evs_handle h, evs_stats_t *out, int reset) {
    if (h == nullptr || out == nullptr) return EVS_ERR_INVALID;
    EVS_CUDA(cudaSetDevice(h->cfg.device));
    EVS_CUDA(cudaDeviceSynchronize());
    GlobalCtl g;
    EVS_CUDA(cudaMemcpy(&g, h->g, sizeof(g), cudaMemcpyDeviceToHost));
    memset(out, 0, sizeof(*out));
    out->lookups = g.lookups;
    out->samples = g.samples;
    out->hits[0] = g.hits[0];
    out->hits[1] = g.hits[1];
    out->c3_hits = g.c3_hits;
    out->approx_subst = g.approx_subst;
    out->misses = g.misses;
    out->perfect_hits = g.perfect_hits;
    out->batches = g.batches;
    for (int i = 0; i < h->n_tiers; ++i) {
        TierCtl c;
        EVS_CUDA(cudaMemcpy(&c, h->tier[i].dev.ctl, sizeof(c), cudaMemcpyDeviceToHost));
        out->inserts[i] = c.stat_inserts;
        out->evictions[i] = c.stat_evictions;
        out->flushed[i] = c.stat_flushed;
        uint64_t sz = 0;
        for (int b = 0; b < h->tier[i].dev.n_buckets; ++b) sz += c.count[b];
        out->size[i] = sz;
        out->capacity[i] = h->tier[i].dev.cap;
        if (reset) {
            c.stat_inserts = c.stat_evictions = c.stat_flushed = 0;
            EVS_CUDA(cudaMemcpy(h->tier[i].dev.ctl, &c, sizeof(c), cudaMemcpyHostToDevice));
        }
    }
    if (h->c3_active) {
        C3Ctl c3;
        EVS_CUDA(cudaMemcpy(&c3, h->params.c3.ctl, sizeof(c3), cudaMemcpyDeviceToHost));
        out->c3_size = c3.size;
        out->c3_capacity = h->params.c3.cap;
    }
    if (reset) {
        const unsigned err = g.error, fds = g.fetch_done_seq, as = g.auto_seq;
        memset(&g, 0, sizeof(g));
        g.error = err;
        g.fetch_done_seq = fds;
        g.auto_seq = as;
        EVS_CUDA(cudaMemcpy(h->g, &g, sizeof(g), cudaMemcpyHostToDevice));
    }
    return EVS_OK;
}

int evs_set_profiling(evs_handle h, int enable) {
    if (h == nullptr) return EVS_ERR_INVALID;
    h->prof.drain();
    h->prof.on = enable != 0;
    return EVS_OK;
}

int evs_kernel_times(evs_handle h, int32_t *n, const char **names, double *total_ms, uint64_t *timed,
                     uint64_t *launches, int reset) {
    if (h == nullptr || n == nullptr) return EVS_ERR_INVALID;
    EVS_CUDA(cudaSetDevice(h->cfg.device));
    h->prof.drain();
    const int cap = *n;
    *n = K_COUNT;
    for (int i = 0; i < K_COUNT && i < cap; ++i) {
        if (names) names[i] = kKernelNames[i];
        if (total_ms) total_ms[i] = h->prof.ms[i];
        if (timed) timed[i] = h->prof.timed[i];
        if (launches) launches[i] = h->prof.launches[i];
    }
    if (reset)
        for (int i = 0; i < K_COUNT; ++i) h->prof.ms[i] = 0.0, h->prof.timed[i] = 0, h->prof.launches[i] = 0;
    return EVS_OK;
}

int evs_phase_times(evs_handle h, uint64_t *ns8) {
    if (h == nullptr || ns8 == nullptr) return EVS_ERR_INVALID;
    EVS_CUDA(cudaSetDevice(h->cfg.device));
    EVS_CUDA(cudaDeviceSynchronize());
    EVS_CUDA(cudaMemcpy(ns8, h->params.dbg, 32 * sizeof(uint64_t), cudaMemcpyDeviceToHost));
    unsigned long long sc = 0, ap = 0;
    EVS_CUDA(cudaMemcpyFromSymbol(&sc, p_dbg_scanned, sizeof(sc)));
    EVS_CUDA(cudaMemcpyFromSymbol(&ap, p_dbg_appends, sizeof(ap)));
    ns8[15] = sc;
    ns8[1] = ap;
    EVS_CUDA(cudaMemset(h->params.dbg + 8, 0, 7 * sizeof(uint64_t)));
    EVS_CUDA(cudaMemset(h->params.dbg + 20, 0, 12 * sizeof(uint64_t)));
    return EVS_OK;
}

uint64_t evs_launch_count(evs_handle h) {
    if (h == nullptr) return 0;
    uint64_t t = 0;
    for (int i = 0; i < K_COUNT; ++i) t += h->prof.launches[i];
    return t;
}

int evs_last_events(evs_handle h, int tier, int64_t *evicted, int64_t *n_evicted, int64_t *flushed, int64_t *n_flushed) {
    if (h == nullptr || tier < 0 || tier >= h->n_tiers || n_evicted == nullptr || n_flushed == nullptr) return EVS_ERR_INVALID;
    EVS_CUDA(cudaSetDevice(h->cfg.device));
    EVS_CUDA(cudaDeviceSynchronize());
    TierCtl c;
    const TierDev &d = h->tier[tier].dev;
    EVS_CUDA(cudaMemcpy(&c, d.ctl, sizeof(c), cudaMemcpyDeviceToHost));
    if (c.n_evicted_last > *n_evicted || c.n_flushed_last > *n_flushed) {
        set_error("evs_last_events: arrays too small");
        return EVS_ERR_INVALID;
    }
    *n_evicted = c.n_evicted_last;
    if (c.n_evicted_last) EVS_CUDA(cudaMemcpy(evicted, d.evicted, sizeof(int64_t) * c.n_evicted_last, cudaMemcpyDeviceToHost));
    if (c.n_flushed_last && d.flushed == nullptr) {
        set_error("evs_last_events: create the handle with record_events to read flushed keys");
        return EVS_ERR_INVALID;
    }
    *n_flushed = c.n_flushed_last;
    if (c.n_flushed_last) EVS_CUDA(cudaMemcpy(flushed, d.flushed, sizeof(int64_t) * c.n_flushed_last, cudaMemcpyDeviceToHost));
    return EVS_OK;
}

// ---- snapshots of the policy state (evs_state.cuh) ---------------------------------------------------------------
// Blob = StateHeader, then per tier: n_perfect, count[n_buckets], the keys bucket by bucket (FIFO order); then, with three
// layers: C3's size, the window length W, the W records, and size map entries (key, alt | flag << 32).  u64 words, little
// endian (include/evstore_b200.h).
struct StateHeader {
    char magic[8];                           // "EVSSTATE"
    uint32_t version, header_bytes;
    uint64_t total_bytes;
    int32_t policy, n_layers, n_tables_total, n_tables;
    int32_t dim, main_precision, secondary_precision, n_buckets;   // precisions and capacities: informational
    uint64_t cap[EVS_MAX_TIERS], c3_cap;
    int32_t table_ids[EVS_MAX_TABLES];       // unused entries -1
    int64_t rows[EVS_MAX_TABLES];            // unused entries 0
};
static_assert(sizeof(StateHeader) == 464 && sizeof(StateHeader) % 8 == 0, "snapshot header layout");
static const char kStateMagic[8] = {'E', 'V', 'S', 'S', 'T', 'A', 'T', 'E'};
constexpr uint32_t kStateVersion = 1;

// Upper bound of the body's words: every tier full, C3 full with a full ring window.
static unsigned long long state_body_bound(evs_handle h) {
    unsigned long long w = 0;
    for (int t = 0; t < h->n_tiers; ++t) w += 1ull + h->tier[t].dev.n_buckets + h->tier[t].dev.cap;
    if (h->c3_active) w += 2ull + h->params.c3.ring_cap + 2ull * h->params.c3.cap;
    return w;
}

static int state_reserve(evs_handle h, unsigned long long body_words) {
    const size_t need = kStateMetaWords + body_words;
    if (need <= h->state_words) return EVS_OK;
    EVS_CUDA(cudaDeviceSynchronize());                        // an earlier call's kernels may still use the buffer
    if (h->state_buf) cudaFree(h->state_buf);
    h->hbm_bytes -= h->state_words * sizeof(unsigned long long);
    h->state_buf = nullptr;
    h->state_words = 0;
    EVS_CUDA(cudaMalloc(&h->state_buf, need * sizeof(unsigned long long)));
    h->state_words = need;
    h->hbm_bytes += need * sizeof(unsigned long long);
    return EVS_OK;
}

static bool state_capturing(cudaStream_t st) {
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    return cudaStreamIsCapturing(st, &cs) == cudaSuccess && cs != cudaStreamCaptureStatusNone;
}

// k_state_save on st, then a synchronise: meta[0] = body words, meta[1] = status, meta[2 + 32 t + b] = live records.
static int state_stage(evs_handle h, cudaStream_t st, unsigned long long (&meta)[kStateMetaWords], const char *what) {
    int rc = state_reserve(h, state_body_bound(h));
    if (rc) return rc;
    EVS_CUDA(cudaMemsetAsync(h->state_buf, 0, kStateMetaWords * sizeof(unsigned long long), st));
    {
        LaunchScope ls(h->prof, K_STATE, st);
        const int ctas = h->n_tiers * h->tier[0].dev.n_buckets + (h->c3_active ? 1 : 0);
        k_state_save<<<ctas, kStateThreads, 0, st>>>(h->params, h->state_buf);
        EVS_CUDA(cudaGetLastError());
    }
    EVS_CUDA(cudaMemcpyAsync(meta, h->state_buf, sizeof(meta), cudaMemcpyDeviceToHost, st));
    EVS_CUDA(cudaStreamSynchronize(st));
    if (meta[1] & kStateOverCap) {
        set_error(std::string(what) + ": a tier holds more keys than its capacity");
        return EVS_ERR_CAPACITY;
    }
    return EVS_OK;
}

static int state_c3_ok(const unsigned long long (&meta)[kStateMetaWords], const char *what) {
    if (!(meta[1] & kStateBadC3)) return EVS_OK;
    set_error(std::string(what) + ": C3's map entries differ from its size");
    return EVS_ERR_CAPACITY;
}

// The body words of tier `tier` (n_perfect, count[], keys) within the staged body.
static size_t state_tier_offset(evs_handle h, const std::vector<unsigned long long> &body, int tier) {
    size_t o = 0;
    for (int t = 0; t < tier; ++t) {
        const int nb = h->tier[t].dev.n_buckets;
        unsigned long long n = 0;
        for (int b = 0; b < nb; ++b) n += body[o + 1 + b];
        o += 1 + nb + n;
    }
    return o;
}

static int state_fetch_body(evs_handle h, cudaStream_t st, const unsigned long long (&meta)[kStateMetaWords], void *dst) {
    if (meta[0]) EVS_CUDA(cudaMemcpyAsync(dst, h->state_buf + kStateMetaWords, meta[0] * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    EVS_CUDA(cudaStreamSynchronize(st));
    return EVS_OK;
}

int evs_state_bytes(evs_handle h, uint64_t *bound) {
    if (h == nullptr || bound == nullptr) return EVS_ERR_INVALID;
    *bound = sizeof(StateHeader) + state_body_bound(h) * sizeof(unsigned long long);
    return EVS_OK;
}

int evs_save_state(evs_handle h, void *buf, uint64_t cap, uint64_t *bytes, void *stream) {
    if (h == nullptr || buf == nullptr || bytes == nullptr) {
        set_error("evs_save_state: bad handle / pointers");
        return EVS_ERR_INVALID;
    }
    DeviceGuard dg(h->cfg.device);
    cudaStream_t st = stream_of(h, stream);
    if (state_capturing(st)) {
        set_error("evs_save_state: the stream is being captured; call it outside a graph, between launches");
        return EVS_ERR_INVALID;
    }
    unsigned long long meta[kStateMetaWords];
    int rc = state_stage(h, st, meta, "evs_save_state");
    if (rc) return rc;
    if (meta[1] & kStateBadBucket) {
        set_error("evs_save_state: a bucket's live records differ from its count");
        return EVS_ERR_CAPACITY;
    }
    if ((rc = state_c3_ok(meta, "evs_save_state"))) return rc;
    const uint64_t total = sizeof(StateHeader) + meta[0] * sizeof(unsigned long long);
    *bytes = total;
    if (cap < total) {
        set_error("evs_save_state: buffer of " + std::to_string(cap) + " B, the snapshot needs " + std::to_string(total) + " B");
        return EVS_ERR_INVALID;
    }
    StateHeader hd{};
    memcpy(hd.magic, kStateMagic, 8);
    hd.version = kStateVersion;
    hd.header_bytes = sizeof(StateHeader);
    hd.total_bytes = total;
    hd.policy = h->cfg.policy;
    hd.n_layers = h->cfg.n_layers;
    hd.n_tables_total = h->cfg.n_tables_total;
    hd.n_tables = h->cfg.n_tables;
    hd.dim = h->cfg.dim;
    hd.main_precision = h->tier[0].prec;
    hd.secondary_precision = h->n_tiers == 2 ? h->tier[1].prec : 0;
    hd.n_buckets = h->tier[0].dev.n_buckets;
    for (int t = 0; t < h->n_tiers; ++t) hd.cap[t] = h->tier[t].dev.cap;
    hd.c3_cap = h->c3_active ? h->params.c3.cap : 0;
    for (int t = 0; t < EVS_MAX_TABLES; ++t) {
        hd.table_ids[t] = t < h->cfg.n_tables ? h->table_ids[t] : -1;
        hd.rows[t] = t < h->cfg.n_tables ? h->rows[t] : 0;
    }
    memcpy(buf, &hd, sizeof(hd));
    return state_fetch_body(h, st, meta, static_cast<unsigned char *>(buf) + sizeof(StateHeader));
}

// Parses and checks a snapshot against the handle on the host; fills the load arguments (offsets into the body).
static int state_parse(evs_handle h, const unsigned char *buf, uint64_t bytes, StateLoadArgs &a, size_t &body_words,
                       size_t &win_off, size_t &map_off) {
    auto bad = [](const std::string &m) {
        set_error("evs_load_state: " + m);
        return EVS_ERR_INVALID;
    };
    if (bytes < sizeof(StateHeader)) return bad("truncated: " + std::to_string(bytes) + " B is shorter than the header");
    StateHeader hd;
    memcpy(&hd, buf, sizeof(hd));
    if (memcmp(hd.magic, kStateMagic, 8) != 0) return bad("not a snapshot (bad magic)");
    if (hd.version != kStateVersion || hd.header_bytes != sizeof(StateHeader))
        return bad("unsupported snapshot version " + std::to_string(hd.version));
    if (hd.total_bytes != bytes) return bad("length " + std::to_string(bytes) + " B, the header says " + std::to_string(hd.total_bytes) + " B");
    if ((bytes - sizeof(StateHeader)) % 8 != 0) return bad("the body is not a whole number of 8-byte words");
    if (hd.policy != h->cfg.policy) return bad("policy " + std::to_string(hd.policy) + " != " + std::to_string(h->cfg.policy));
    if (hd.n_layers != h->cfg.n_layers) return bad("n_layers " + std::to_string(hd.n_layers) + " != " + std::to_string(h->cfg.n_layers));
    if (hd.n_tables_total != h->cfg.n_tables_total) return bad("n_tables_total differs");
    if (hd.n_tables != h->cfg.n_tables || hd.n_buckets != h->tier[0].dev.n_buckets) return bad("the served tables differ");
    for (int t = 0; t < h->cfg.n_tables; ++t) {
        if (hd.table_ids[t] != h->table_ids[t]) return bad("the served tables differ");
        if (hd.rows[t] != h->rows[t]) return bad("rows of table " + std::to_string(h->table_ids[t]) + " differ");
    }
    const unsigned long long *w = reinterpret_cast<const unsigned long long *>(buf + sizeof(StateHeader));
    const size_t nw = (bytes - sizeof(StateHeader)) / 8;
    size_t o = 0;
    const int nb = h->tier[0].dev.n_buckets;
    a = StateLoadArgs{};
    for (int t = 0; t < h->n_tiers; ++t) {
        if (o + 1 + nb > nw) return bad("truncated in tier " + std::to_string(t));
        if (w[o] > 0xFFFFFFFFull) return bad("n_perfect out of range");
        a.n_perfect[t] = static_cast<unsigned>(w[o]);
        unsigned long long n = 0;
        a.off[t][0] = 0;
        for (int b = 0; b < nb; ++b) {
            n += w[o + 1 + b];
            if (n > h->tier[t].dev.cap)
                return bad("tier " + std::to_string(t) + " holds more keys than this handle's capacity " + std::to_string(h->tier[t].dev.cap));
            a.off[t][b + 1] = static_cast<unsigned>(n);
        }
        o += 1 + nb;
        if (o + n > nw) return bad("truncated in tier " + std::to_string(t));
        a.keys[t] = reinterpret_cast<const unsigned long long *>(o * 8);      // offset; the device address is added later
        o += n;
    }
    win_off = map_off = 0;
    if (h->c3_active) {
        if (o + 2 > nw) return bad("truncated in C3");
        const unsigned long long size = w[o], W = w[o + 1];
        const unsigned long long c3cap = h->params.c3.cap, ring = h->params.c3.ring_cap;
        if (size > c3cap) return bad("C3 holds " + std::to_string(size) + " keys, more than this handle's capacity " + std::to_string(c3cap));
        // the next batch's c3_update appends up to the victims of both tiers behind the window (evs_c3.cuh)
        const unsigned long long room = 2ull * static_cast<unsigned long long>(h->cfg.max_batch) * h->cfg.n_tables;
        if (W + room > ring)
            return bad("C3's window of " + std::to_string(W) + " records leaves no room for a batch's " + std::to_string(room) +
                       " appends in this handle's ring of " + std::to_string(ring));
        o += 2;
        if (o + W + 2 * size > nw) return bad("truncated in C3");
        win_off = o;
        a.W = W;
        o += W;
        map_off = o;
        a.n_map = static_cast<unsigned>(size);
        o += 2 * size;
    }
    if (o != nw) return bad("the body has " + std::to_string(nw) + " words, its sections " + std::to_string(o));
    body_words = nw;
    return EVS_OK;
}

// Clears every tier and C3 and, with a = the parsed snapshot, loads it (k_init_* -> k_state_load[_c3] -> k_state_load_ctl).
static int state_install(evs_handle h, cudaStream_t st, const StateLoadArgs &a, bool load) {
    LaunchScope ls(h->prof, K_STATE, st);
    for (int t = 0; t < h->n_tiers; ++t) k_init_tier<<<592, 256, 0, st>>>(h->tier[t].dev);
    if (h->c3_active) k_init_c3<<<592, 256, 0, st>>>(h->params.c3);
    EVS_CUDA(cudaGetLastError());
    // no programmatic serialization: the next batch's k_serve cannot start before the state is complete
    void *args[] = {&h->params, const_cast<StateLoadArgs *>(&a)};
    if (load) {
        const unsigned n = a.off[0][h->tier[0].dev.n_buckets] + (h->n_tiers == 2 ? a.off[1][h->tier[1].dev.n_buckets] : 0u);
        if (n) EVS_CUDA(launch_ex(reinterpret_cast<const void *>(k_state_load), dim3(std::min<unsigned>((n + 7) / 8, 148 * 16)), 256, 0, st, args, false));
        if (h->c3_active && a.n_map + a.W)
            EVS_CUDA(launch_ex(reinterpret_cast<const void *>(k_state_load_c3), dim3(static_cast<unsigned>(std::min<unsigned long long>((a.n_map + a.W + 255) / 256, 148 * 8))),
                               256, 0, st, args, false));
    }
    EVS_CUDA(launch_ex(reinterpret_cast<const void *>(k_state_load_ctl), dim3(1), 32, 0, st, args, false));
    return EVS_OK;
}

int evs_load_state(evs_handle h, const void *buf, uint64_t bytes, void *stream) {
    if (h == nullptr || buf == nullptr) {
        set_error("evs_load_state: bad handle / pointer");
        return EVS_ERR_INVALID;
    }
    DeviceGuard dg(h->cfg.device);
    cudaStream_t st = stream_of(h, stream);
    if (state_capturing(st)) {
        set_error("evs_load_state: the stream is being captured; call it outside a graph, between launches");
        return EVS_ERR_INVALID;
    }
    StateLoadArgs a;
    size_t body_words = 0, win_off = 0, map_off = 0;
    int rc = state_parse(h, static_cast<const unsigned char *>(buf), bytes, a, body_words, win_off, map_off);
    if (rc) return rc;
    if ((rc = state_reserve(h, body_words))) return rc;
    if (h->ev_upd == nullptr) EVS_CUDA(cudaEventCreateWithFlags(&h->ev_upd, cudaEventDisableTiming));
    unsigned long long *body = h->state_buf + kStateMetaWords;
    EVS_CUDA(cudaMemsetAsync(h->state_buf, 0, kStateMetaWords * sizeof(unsigned long long), st));
    if (body_words)
        EVS_CUDA(cudaMemcpyAsync(body, static_cast<const unsigned char *>(buf) + sizeof(StateHeader), body_words * 8, cudaMemcpyHostToDevice, st));
    for (int t = 0; t < h->n_tiers; ++t) a.keys[t] = body + reinterpret_cast<uintptr_t>(a.keys[t]) / 8;
    a.window = body + win_off;
    a.map = body + map_off;
    a.err = reinterpret_cast<unsigned *>(h->state_buf + 1);
    if ((rc = state_install(h, st, a, true))) return rc;
    // the look-ahead: an announcement made before the load staged rows of the old state's misses -- cancel it, and order
    // every later k_prefetch behind the new state (as evs_update_rows does)
    h->pf.cancel();
    EVS_CUDA(cudaEventRecord(h->ev_upd, st));
    EVS_CUDA(cudaStreamWaitEvent(h->pf_stream, h->ev_upd, 0));
    unsigned long long err = 0;
    EVS_CUDA(cudaMemcpyAsync(&err, h->state_buf + 1, sizeof(err), cudaMemcpyDeviceToHost, st));
    EVS_CUDA(cudaStreamSynchronize(st));
    if (err) {
        StateLoadArgs empty{};
        if ((rc = state_install(h, st, empty, false))) return rc;
        EVS_CUDA(cudaStreamSynchronize(st));
    }
    // the ring-occupancy mirror (maintain_rings): the device is idle, the rings hold count records from position 0
    for (int t = 0; t < h->n_tiers; ++t) {
        unsigned long long mx = 0;
        if (!err)
            for (int b = 0; b < h->tier[t].dev.n_buckets; ++b) mx = std::max<unsigned long long>(mx, a.off[t][b + 1] - a.off[t][b]);
        *reinterpret_cast<volatile unsigned long long *>(h->ring_host + t) = (static_cast<unsigned long long>(static_cast<unsigned>(h->seq)) << 32) | mx;
    }
    if (err) {
        set_error(std::string("evs_load_state: ") + ((err & kStateBadKey) ? "a key's table is not served here or its row is out of range"
                                                                            : "a key appears twice in one tier or in C3's map") +
                  "; the handle is now empty");
        return EVS_ERR_INVALID;
    }
    return EVS_OK;
}

int evs_dump_state(evs_handle h, int tier, int64_t *keys, int64_t *n_keys, int64_t *bucket_off, int64_t *n_perfect) {
    if (h == nullptr || tier < 0 || tier >= h->n_tiers || keys == nullptr || n_keys == nullptr || bucket_off == nullptr)
        return EVS_ERR_INVALID;
    EVS_CUDA(cudaSetDevice(h->cfg.device));
    EVS_CUDA(cudaDeviceSynchronize());
    unsigned long long meta[kStateMetaWords];
    int rc = state_stage(h, h->stream, meta, "evs_dump_state");
    if (rc) return rc;
    std::vector<unsigned long long> body(meta[0]);
    if ((rc = state_fetch_body(h, h->stream, meta, body.data()))) return rc;
    const int nb = h->tier[tier].dev.n_buckets;
    const size_t o = state_tier_offset(h, body, tier);
    int64_t n = 0;
    for (int b = 0; b < nb; ++b) {
        const unsigned long long cnt = body[o + 1 + b], live = meta[2 + kMaxBuckets * tier + b];
        if (live != cnt) {
            set_error("evs_dump_state: bucket " + std::to_string(b) + " live records " + std::to_string(live) + " != count " + std::to_string(cnt));
            return EVS_ERR_CAPACITY;
        }
        bucket_off[b] = n;
        if (n + static_cast<int64_t>(cnt) > *n_keys) {
            set_error("evs_dump_state: keys array too small");
            return EVS_ERR_INVALID;
        }
        for (unsigned long long i = 0; i < cnt; ++i) keys[n + i] = static_cast<int64_t>(body[o + 1 + nb + n + i]);
        n += static_cast<int64_t>(cnt);
    }
    bucket_off[nb] = n;
    *n_keys = n;
    if (n_perfect) *n_perfect = static_cast<int64_t>(body[o]);
    return EVS_OK;
}

// C3 in FIFO order: one entry per queue record whose key is still mapped (stale records of
// evicted keys are skipped, duplicates of a mapped key are reported as they sit in the queue).
int evs_dump_c3(evs_handle h, int64_t *keys, uint32_t *alt, uint8_t *recency, int64_t *n) {
    if (h == nullptr || n == nullptr) return EVS_ERR_INVALID;
    if (!h->c3_active) {
        *n = 0;
        return EVS_OK;
    }
    EVS_CUDA(cudaSetDevice(h->cfg.device));
    EVS_CUDA(cudaDeviceSynchronize());
    unsigned long long meta[kStateMetaWords];
    int rc = state_stage(h, h->stream, meta, "evs_dump_c3");
    if (rc || (rc = state_c3_ok(meta, "evs_dump_c3"))) return rc;
    std::vector<unsigned long long> body(meta[0]);
    if ((rc = state_fetch_body(h, h->stream, meta, body.data()))) return rc;
    const size_t o = state_tier_offset(h, body, h->n_tiers);
    const unsigned long long size = body[o], W = body[o + 1];
    const unsigned long long *win = body.data() + o + 2, *map = win + W;
    std::map<unsigned long long, unsigned long long> mapped;
    for (unsigned long long i = 0; i < size; ++i) mapped[map[2 * i]] = map[2 * i + 1];
    int64_t cnt = 0;
    for (unsigned long long q = 0; q < W; ++q) {
        const auto it = mapped.find(win[q]);
        if (it == mapped.end()) continue;
        if (cnt >= *n) {
            set_error("evs_dump_c3: arrays too small");
            return EVS_ERR_INVALID;
        }
        if (keys) keys[cnt] = static_cast<int64_t>(win[q]);
        if (alt) alt[cnt] = static_cast<uint32_t>(it->second);
        if (recency) recency[cnt] = static_cast<uint8_t>((it->second >> 32) & 1u);
        ++cnt;
    }
    *n = cnt;
    return EVS_OK;
}

int evs_interact(const float *x_dev, const float *ly_dev, float *r_dev, int32_t B, int32_t n_f, int32_t dim, void *stream) {
    return launch_interact(x_dev, ly_dev, r_dev, B, n_f, dim, static_cast<cudaStream_t>(stream));
}

// ---- table-wise sharding over NVLink peer memory -----------------------------------------------
// First 256 bytes of every rank's exchange block: what the rank was built with, so that evs_shard_connect can refuse
// a peer whose layout differs (rows would otherwise land at the wrong offsets of its receive buffer).
struct ShardHeader {
    unsigned magic, world, rank, t_total, dim, batch_max;
    unsigned table_mask;                      // bit g: this rank serves global table g
};
constexpr unsigned kShardMagic = 0x45565332u;  // "EVS2"

int evs_shard_create(evs_handle h, int32_t rank, int32_t world, int32_t batch_max, evs_shard *out) {
    if (h == nullptr || out == nullptr || world < 1 || world > kMaxPeers || rank < 0 || rank >= world || batch_max < world ||
        batch_max % world != 0 || batch_max > h->cfg.max_batch) {
        set_error("evs_shard_create: bad rank / world / batch_max (batch_max must be a multiple of world and <= max_batch)");
        return EVS_ERR_INVALID;
    }
    DeviceGuard dg(h->cfg.device);
    evs_shard s = new evs_shard_s();
    s->h = h;
    s->rank = rank;
    s->world = world;
    s->batch_max = batch_max;
    s->t_total = h->cfg.n_tables_total;
    const size_t bl = static_cast<size_t>(batch_max / world);
    s->off_recv = 256;
    s->recv_bytes = (bl * s->t_total * h->cfg.dim * sizeof(float) + 255) & ~static_cast<size_t>(255);
    s->off_parts = s->off_recv + evs_shard_s::kRecvBufs * s->recv_bytes;
    s->off_oflags = (s->off_parts + 2 * sizeof(unsigned) * static_cast<size_t>(world) * batch_max + 255) & ~static_cast<size_t>(255);
    s->bytes = s->off_oflags + 256;
    void *q = nullptr;
    cudaError_t e = cudaMalloc(&q, s->bytes);
    if (e != cudaSuccess) {
        set_error(std::string("evs_shard_create: cudaMalloc -> ") + cudaGetErrorString(e));
        delete s;
        return EVS_ERR_CUDA;
    }
    h->hbm_bytes += s->bytes;
    cudaMemset(q, 0, s->bytes);
    ShardHeader hd{};
    hd.magic = kShardMagic;
    hd.world = static_cast<unsigned>(world);
    hd.rank = static_cast<unsigned>(rank);
    hd.t_total = static_cast<unsigned>(s->t_total);
    hd.dim = static_cast<unsigned>(h->cfg.dim);
    hd.batch_max = static_cast<unsigned>(batch_max);
    for (int g : h->table_ids) hd.table_mask |= 1u << g;
    cudaMemcpy(q, &hd, sizeof(hd), cudaMemcpyHostToDevice);
    cudaDeviceSynchronize();
    s->block = static_cast<unsigned char *>(q);
    s->peer[rank] = s->block;
    *out = s;
    return EVS_OK;
}

int evs_shard_export(evs_shard s, void *handle64) {
    if (s == nullptr || handle64 == nullptr) return EVS_ERR_INVALID;
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
    DeviceGuard dg(s->h->cfg.device);
    cudaIpcMemHandle_t hd;
    EVS_CUDA(cudaIpcGetMemHandle(&hd, s->block));
    memcpy(handle64, &hd, sizeof(hd));
    return EVS_OK;
}

int evs_shard_connect(evs_shard s, const void *handles) {
    if (s == nullptr || handles == nullptr) return EVS_ERR_INVALID;
    DeviceGuard dg(s->h->cfg.device);
    evs_handle h = s->h;
    unsigned seen = 0;
    for (int r = 0; r < s->world; ++r) {
        if (r != s->rank) {
            cudaIpcMemHandle_t hd;
            memcpy(&hd, static_cast<const unsigned char *>(handles) + 64 * r, sizeof(hd));
            void *q = nullptr;
            cudaError_t e = cudaIpcOpenMemHandle(&q, hd, cudaIpcMemLazyEnablePeerAccess);
            if (e != cudaSuccess) {
                set_error("evs_shard_connect: cudaIpcOpenMemHandle(rank " + std::to_string(r) + ") -> " + cudaGetErrorString(e));
                cudaGetLastError();
                return EVS_ERR_CUDA;
            }
            s->peer[r] = static_cast<unsigned char *>(q);
            s->opened[r] = true;
        }
        // every rank must have been built for the same model and exchange layout, and no table may be served twice
        ShardHeader ph{};
        EVS_CUDA(cudaMemcpy(&ph, s->peer[r], sizeof(ph), cudaMemcpyDeviceToHost));
        if (ph.magic != kShardMagic || ph.world != static_cast<unsigned>(s->world) || ph.rank != static_cast<unsigned>(r) ||
            ph.t_total != static_cast<unsigned>(s->t_total) || ph.dim != static_cast<unsigned>(h->cfg.dim) ||
            ph.batch_max != static_cast<unsigned>(s->batch_max) || (ph.table_mask & seen) != 0u) {
            set_error("evs_shard_connect: rank " + std::to_string(r) + " was created with a different world / n_tables_total / dim / "
                      "batch_max, or serves a table another rank serves");
            return EVS_ERR_INVALID;
        }
        seen |= ph.table_mask;
    }
    // from here on the batch is k_serve<.., true> ... k_evict with the peer completion in its tail, and a table's rows
    // go to the column of its global id in the owner ranks' receive buffers
    EVS_CUDA(cudaDeviceSynchronize());
    h->sharded = true;
    for (int t = 0; t < h->cfg.n_tables; ++t) h->params.col[t] = h->table_ids[t];
    // one-pass exchange needs every CTA of k_serve co-resident (they spin on words the peers' last CTAs raise)
    {
        const KernelSet ks = kernels_of_handle(h);
        int per_sm = 0, sms = 0;
        EVS_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, reinterpret_cast<const void *>(ks.serve_sh), kLookupThreads, 0));
        EVS_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, h->cfg.device));
        const int n_chunks = (s->batch_max + h->params.spc - 1) / h->params.spc;
        // half of the slots at most: the look-ahead kernel and the caller's own kernels may hold the others
        s->fused = n_chunks <= per_sm * sms / 2;
        const char *nf = getenv("EVSTORE_B200_SHARD_TWO_PASS");    // tuning aid: 1 = separate probe pass (the round-1 path)
        if (nf && nf[0] == '1') s->fused = false;
    }
    if (h->use_graph) {
        destroy_graphs(h);
        int rc = build_graph(h);
        if (rc) return rc;
    }
    return EVS_OK;
}

// The exchange arguments of the batch with number `epoch`: receive buffer epoch % kRecvBufs of every rank, count table epoch % 2.
static ShardArgs shard_args(evs_shard s, int32_t B, unsigned epoch) {
    ShardArgs sh{};
    sh.world = s->world;
    sh.rank = s->rank;
    sh.Bl = B / s->world;
    sh.T_total = s->t_total;
    sh.epoch = epoch;
    sh.fused = s->fused ? 1 : 0;
    const unsigned par = epoch & 1u, buf = epoch % evs_shard_s::kRecvBufs;
    const size_t parts_par = s->off_parts + sizeof(unsigned) * static_cast<size_t>(par) * s->world * s->batch_max;
    for (int r = 0; r < s->world; ++r) {
        sh.recv[r] = reinterpret_cast<float *>(s->peer[r] + s->off_recv + buf * s->recv_bytes);
        sh.parts[r] = reinterpret_cast<unsigned *>(s->peer[r] + parts_par) + static_cast<size_t>(s->rank) * B;
        sh.out_flag[r] = reinterpret_cast<unsigned *>(s->peer[r] + s->off_oflags) + s->rank;
    }
    sh.my_parts = reinterpret_cast<const unsigned *>(s->block + parts_par);
    sh.my_out_flags = reinterpret_cast<const unsigned *>(s->block + s->off_oflags);
    return sh;
}

static int shard_check(evs_shard s, const char *what, int32_t B) {
    if (s == nullptr || B < s->world || B > s->batch_max || B % s->world != 0) {
        set_error(std::string(what) + ": bad shard / B (B must be a multiple of world, <= batch_max)");
        return EVS_ERR_INVALID;
    }
    for (int r = 0; r < s->world; ++r)
        if (s->peer[r] == nullptr) {
            set_error(std::string(what) + ": evs_shard_connect has not been called");
            return EVS_ERR_NOT_CONFIGURED;
        }
    return EVS_OK;
}

// n consecutive global batches on this rank: batch i takes the next exchange epoch and gets that epoch's receive buffer,
// which out_dev[i] reports; without the one-pass exchange a probe pass goes ahead of each batch.  The receive buffers
// rotate through kRecvBufs = 4, so a buffer is valid until four batches later.
static int shard_submit(evs_shard s, cudaStream_t st, int32_t n, const int64_t *const *idx_dev, int32_t B, uint8_t *const *hit_dev,
                        float **out_dev) {
    evs_handle h = s->h;
    return submit_batches(h, st, n, idx_dev, B, s->fused, [&](int i, BatchArgs &a) {
        const unsigned epoch = ++s->epoch;
        a = lookup_args(h, idx_dev[i], B, nullptr, 0, hit_dev ? hit_dev[i] : nullptr);
        a.sh = shard_args(s, B, epoch);
        out_dev[i] = reinterpret_cast<float *>(s->block + s->off_recv + (epoch % evs_shard_s::kRecvBufs) * s->recv_bytes);
        return s->fused ? EVS_OK : launch_probe(h, a, st);
    });
}

int evs_shard_lookup(evs_shard s, const int64_t *idx_dev, int32_t B, uint8_t *hit_dev, float **out_dev, void *stream) {
    if (idx_dev == nullptr || out_dev == nullptr) {
        set_error("evs_shard_lookup: null pointer");
        return EVS_ERR_INVALID;
    }
    int rc = shard_check(s, "evs_shard_lookup", B);
    if (rc) return rc;
    DeviceGuard dg(s->h->cfg.device);
    return shard_submit(s, stream_of(s->h, stream), 1, &idx_dev, B, &hit_dev, out_dev);
}

// n consecutive global batches in one call (evs_lookup_batches for a rank of a sharded cache): with the one-pass exchange,
// groups of 4 batches go to the device as one captured graph on every rank.
int evs_shard_lookup_many(evs_shard s, int32_t n, const int64_t *const *idx_dev, int32_t B, uint8_t *const *hit_dev, float **out_dev,
                          void *stream) {
    if (n < 0 || (n > 0 && (idx_dev == nullptr || out_dev == nullptr))) {
        set_error("evs_shard_lookup_many: bad n / pointers");
        return EVS_ERR_INVALID;
    }
    int rc = shard_check(s, "evs_shard_lookup_many", B);
    if (rc) return rc;
    DeviceGuard dg(s->h->cfg.device);
    return shard_submit(s, stream_of(s->h, stream), n, idx_dev, B, hit_dev, out_dev);
}

// Bags on a rank of a sharded cache: the rank's tables' bags of the whole global batch as B*P slices whose agg_hit counts
// go through the exchange (fused or a separate probe pass, as for a plain batch); the slice rows stay in the handle's
// staging, and k_bags_pool sends the pooled rows to the owner ranks and closes the epoch.  One batch per call: no
// grouping, no look-ahead.  Plain and bags batches share the epoch sequence and the four receive buffers.
int evs_shard_lookup_bags(evs_shard s, const int64_t *idx_dev, const int64_t *off_dev, int32_t B, int64_t nnz, int32_t max_per_bag,
                          uint8_t *hit_dev, float **out_dev, void *stream) {
    if (s == nullptr || out_dev == nullptr) {
        set_error("evs_shard_lookup_bags: null pointer");
        return EVS_ERR_INVALID;
    }
    int rc = bags_check(s->h, "evs_shard_lookup_bags", idx_dev, off_dev, B, nnz, max_per_bag, s->batch_max);
    if (rc || (rc = shard_check(s, "evs_shard_lookup_bags", B))) return rc;
    evs_handle h = s->h;
    DeviceGuard dg(h->cfg.device);
    cudaStream_t st = stream_of(h, stream);
    const int P = max_per_bag;
    if ((rc = bags_expand(h, st, idx_dev, off_dev, B, nnz, P))) return rc;
    const unsigned epoch = s->epoch + 1;
    const int64_t *slices = reinterpret_cast<const int64_t *>(h->bag_idx);
    rc = submit_batches(h, st, 1, &slices, B * P, false, [&](int, BatchArgs &a) {
        s->epoch = epoch;
        a = bags_args(h, B, P);
        a.sh = shard_args(s, B * P, epoch);                  // the count tables are indexed by slice
        return s->fused ? EVS_OK : launch_probe(h, a, st);
    });
    if (rc) return rc;
    if ((rc = bags_pool(h, st, shard_args(s, B, epoch), off_dev, B, P, nnz, nullptr, 0, hit_dev))) return rc;   // by pooled sample
    *out_dev = reinterpret_cast<float *>(s->block + s->off_recv + (epoch % evs_shard_s::kRecvBufs) * s->recv_bytes);
    return EVS_OK;
}

int evs_shard_destroy(evs_shard s) {
    if (s == nullptr) return EVS_ERR_INVALID;
    cudaSetDevice(s->h->cfg.device);
    cudaDeviceSynchronize();
    for (int r = 0; r < s->world; ++r)
        if (s->opened[r]) cudaIpcCloseMemHandle(s->peer[r]);
    if (s->block) cudaFree(s->block);
    cudaGetLastError();
    delete s;
    return EVS_OK;
}

// ---- sum-pooling gather (nn.EmbeddingBag(mode="sum")) ----------------------------------------
static unsigned *g_gather_err[64] = {};       // per device: an index was out of range

int evs_embedding_bag(const void *table_dev, int64_t rows, int32_t dim, int32_t precision, const int64_t *idx_dev,
                      const int64_t *off_dev, int64_t nnz, int32_t B, const float *per_sample_weights, float *out_dev,
                      int64_t out_stride, void *stream) {
    int dev = 0;
    EVS_CUDA(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 64) return EVS_ERR_INVALID;
    if (g_gather_err[dev] == nullptr) {
        EVS_CUDA(cudaMalloc(&g_gather_err[dev], sizeof(unsigned)));
        EVS_CUDA(cudaMemset(g_gather_err[dev], 0, sizeof(unsigned)));
    }
    int rc = launch_gather(table_dev, rows, dim, precision, reinterpret_cast<const long long *>(idx_dev),
                           reinterpret_cast<const long long *>(off_dev), nnz, B, per_sample_weights, out_dev, out_stride,
                           g_gather_err[dev], static_cast<cudaStream_t>(stream));
    if (rc == EVS_ERR_INVALID) set_error("evs_embedding_bag: bad table / rows / dim / precision / pointers");
    return rc;
}

int evs_embedding_bag_status(void) {
    int dev = 0;
    EVS_CUDA(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 64 || g_gather_err[dev] == nullptr) return EVS_OK;
    EVS_CUDA(cudaDeviceSynchronize());
    unsigned e = 0;
    EVS_CUDA(cudaMemcpy(&e, g_gather_err[dev], sizeof(e), cudaMemcpyDeviceToHost));
    if (e) {
        EVS_CUDA(cudaMemset(g_gather_err[dev], 0, sizeof(unsigned)));
        set_error("evs_embedding_bag: an index was outside [0, rows)");
        return EVS_ERR_INDEX;
    }
    return EVS_OK;
}

// ---- host memory for backing rows -------------------------------------------------------------
// cudaHostAlloc / cudaHostRegister memory is mapped into the device with 4 KB entries whatever the host pages behind it:
// once the random rows of a batch's misses spread over more than ~512 MB the zero-copy read rate halves
// (profiles/r2_zc_page_probe.txt).  Managed memory whose preferred location is the CPU and that is `accessed by` the
// device stays in host memory, is never migrated, and is mapped with large pages: 240 instead of 120-140 row reads / us over
// a 2 GB table (profiles/r2_zc_vmm_probe.txt).  The host reads and writes it like any allocation.
int evs_host_alloc(void **ptr, uint64_t bytes, int32_t device) {
    if (ptr == nullptr || bytes == 0) return EVS_ERR_INVALID;
    *ptr = nullptr;
    DeviceGuard dg(device);
    void *p = nullptr;
    cudaError_t e = cudaMallocManaged(&p, bytes, cudaMemAttachGlobal);
    if (e != cudaSuccess) {
        set_error(std::string("evs_host_alloc: cudaMallocManaged(") + std::to_string(bytes) + " B) -> " + cudaGetErrorString(e));
        cudaGetLastError();
        return EVS_ERR_CUDA;
    }
    e = cudaMemAdvise(p, bytes, cudaMemAdviseSetPreferredLocation, cudaCpuDeviceId);
    if (e == cudaSuccess) e = cudaMemAdvise(p, bytes, cudaMemAdviseSetAccessedBy, device);
    if (e != cudaSuccess) {
        set_error(std::string("evs_host_alloc: cudaMemAdvise -> ") + cudaGetErrorString(e));
        cudaGetLastError();
        cudaFree(p);
        return EVS_ERR_CUDA;
    }
    *ptr = p;
    return EVS_OK;
}

int evs_host_free(void *ptr) {
    if (ptr == nullptr) return EVS_OK;
    EVS_CUDA(cudaFree(ptr));
    return EVS_OK;
}

// ---- alt-key generation: brute-force k-NN over all embedding rows + most popular neighbour (evs_knn.cuh) ----------------
int evs_knn(const float *x_dev, int64_t n, const float *q_dev, int64_t nq, int32_t dim, int32_t k, int64_t *nbr_dev, float *dist_dev,
            const uint32_t *freq_dev, const int64_t *table_off_dev, int32_t n_tables, uint32_t *alt_dev, void *stream) {
    if (nq < 0 || n < 1) return EVS_ERR_INVALID;
    if (nq == 0) return EVS_OK;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    // few query blocks: split the database over CTAs so that the machine is full (the per-split lists are merged afterwards)
    int sms = 148, dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const long long qblocks = (nq + kKnnQ - 1) / kKnnQ;
    const long long tiles = (n + kKnnT - 1) / kKnnT;
    int splits = static_cast<int>(std::max<long long>(1, std::min<long long>(std::min<long long>(tiles, 64), (2ll * sms + qblocks - 1) / qblocks)));
    float2 *part = nullptr;
    EVS_CUDA(cudaMallocAsync(reinterpret_cast<void **>(&part), static_cast<size_t>(nq) * splits * kKnnSel * sizeof(float2), st));
    int rc = launch_knn(x_dev, n, q_dev, nq, dim, k, reinterpret_cast<long long *>(nbr_dev), dist_dev, freq_dev,
                        reinterpret_cast<const long long *>(table_off_dev), n_tables, alt_dev, part, splits, st);
    cudaFreeAsync(part, st);
    if (rc == EVS_ERR_INVALID) set_error("evs_knn: bad pointers / n (< 2^31) / dim (1..64) / k (1..10)");
    return rc;
}

int evs_store_ptr(evs_handle h, int tier, int table, const void **dev_ptr, int32_t *precision) {
    if (h == nullptr || tier < 0 || tier >= h->n_tiers || table < 0 || table >= h->cfg.n_tables || dev_ptr == nullptr)
        return EVS_ERR_INVALID;
    *dev_ptr = h->tier[tier].store_dev[table];
    if (precision) *precision = h->tier[tier].prec;
    return EVS_OK;
}

// ---- legacy libcachemanager.so surface ----------------------------------------------------
static evs_handle g_legacy = nullptr;
static std::vector<float> g_legacy_out;       // emb_weights_in_1d_floats (cache_manager.hpp:51)
static std::vector<int64_t> g_legacy_idx;
static uint64_t g_legacy_perfect_base = 0, g_legacy_c3_base = 0;

int evs_legacy_configure(const evs_config *cfg) {
    if (g_legacy) {
        evs_destroy(g_legacy);
        g_legacy = nullptr;
    }
    int rc = evs_create(cfg, &g_legacy);
    if (rc) return rc;
    g_legacy_out.assign(static_cast<size_t>(cfg->n_tables) * cfg->dim, 0.0f);
    g_legacy_idx.assign(cfg->n_tables, 0);
    g_legacy_perfect_base = g_legacy_c3_base = 0;
    return EVS_OK;
}

evs_handle evs_legacy_handle(void) { return g_legacy; }

float *ev_lookup(int *arr) {
    if (g_legacy == nullptr) {
        fprintf(stderr, "evstore_b200: ev_lookup before evs_legacy_configure\n");
        return nullptr;
    }
    for (size_t t = 0; t < g_legacy_idx.size(); ++t) g_legacy_idx[t] = arr[t];
    int rc = evs_lookup_batch_host(g_legacy, g_legacy_idx.data(), 1, g_legacy_out.data(), nullptr);
    if (rc) {
        fprintf(stderr, "evstore_b200: ev_lookup failed (%d): %s\n", rc, evs_last_error());
        return nullptr;
    }
    return g_legacy_out.data();
}

float *get_ev_values(int *arr) {
    (void)arr;
    return g_legacy_out.empty() ? nullptr : g_legacy_out.data();
}

void print_perfect_hit(void) {
    if (g_legacy == nullptr) {
        fprintf(stderr, "evstore_b200: print_perfect_hit before evs_legacy_configure\n");
        return;
    }
    evs_stats_t s;
    if (evs_stats(g_legacy, &s, 0)) return;
    const evs_config &c = g_legacy->cfg;
    printf("\n[epoll worker] C1_PRECISION    = %d\n", c.main_precision);
    if (c.n_layers >= 2) printf("[epoll worker] C2_PRECISION    = %d\n", c.secondary_precision);
    if (c.n_layers == 3) {
        printf("[epoll worker] C3 APRX_EV      = ACTIVE\n");
        printf("[epoll worker] SIZE_PROPORTION = %d-%d-%d\n", c.prop_c1, c.prop_c2, c.prop_c3);
        // the reference never resets aprx_ev_hit; keep it cumulative too
        printf("[epoll worker] C3 Indiv-Hit    = %llu\n", static_cast<unsigned long long>(s.c3_hits));
    }
    printf("[epoll worker] TOTAL_SIZE      = %lld\n", static_cast<long long>(c.total_size));
    printf("[epoll worker] Perfect hit     = %llu\n", static_cast<unsigned long long>(s.perfect_hits - g_legacy_perfect_base));
    fflush(stdout);
    g_legacy_perfect_base = s.perfect_hits;   // cache_manager.cpp:289 resets the counter
}

void test_arr(int *arr) {
    for (int i = 0; i < 5; i++) printf("key %d, ", arr[i]);
    printf("\n");
    for (int i = 0; i < 5; i++) printf("vec %d, ", arr[i]);
    printf("\n");
    fflush(stdout);
}

int ev_lookup_based_on_list_keys(int *arr) {
    (void)arr;
    fprintf(stderr, "ERROR: This ev_lookup_based_on_list_keys() is outdated, use ev_lookup() instead!\n");
    return -1;
}

}  // extern "C"
