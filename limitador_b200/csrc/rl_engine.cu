// rl_engine.cu — host side of librl_engine.so: limit registry, device tables, workspace,
// kernel launches and the C-ABI declared in include/rl_engine.h.
//
// There is NO CPU fallback: every entry point either runs the sm_100a kernels or returns
// an error.  The reference path this replaces: limitador/src/storage/in_memory.rs
// (InMemoryStorage) behind trait CounterStorage (limitador/src/storage/mod.rs:279-292).
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <string>
#include <utility>
#include <vector>

#include <functional>

#include "rl_kernels.cuh"
#include "rl_shard.cuh"
#include "rl_internal.h"

#ifndef RL_SETS
#define RL_SETS 3  // RL_FLAG_PIPELINE: calls in flight on the device (>= 3: one per pipeline stage)
#endif
#ifndef RL_RING
#define RL_RING 4  // RL_MEM_HOST_ASYNC: staging slots (H2D of call i+RL_RING waits for the D2H of call i)
#endif

namespace {

constexpr uint32_t kMaxTiles = RL_MAX_TILES;
constexpr uint32_t kMaxRegions = 4096;

struct HostLimit {
    bool defined = false;
    uint32_t ns = 0, varset = 0, qualified = 0;
    uint64_t max_value = 0, window_us = 0;
    uint32_t group = 0, cell = 0;
    bool simple_present = false;  // unqualified: entry exists in simple_limits (in_memory.rs:14)
};
struct HostGroup {
    uint32_t ns = 0, varset = 0, qualified = 0;
    uint32_t limit_of_cell[RL_MAX_CELLS];
    HostGroup() {
        for (auto& l : limit_of_cell) l = RL_NONE_U32;
    }
};

template <class T>
struct DevBuf {
    T* p = nullptr;
    size_t n = 0;
    cudaError_t reserve(size_t want) {
        if (want <= n) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr;
        n = 0;
        cudaError_t r = cudaMalloc((void**)&p, want * sizeof(T));
        if (r == cudaSuccess) n = want;
        return r;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        n = 0;
    }
};

}  // namespace

// A second copy of the per-batch workspace: with RL_FLAG_PIPELINE the partition kernels of
// batch s+1 run (on their own stream) while k_main of batch s is still replaying.
struct WorkSet {
    DevBuf<uint32_t> tile_loc, region_total, part_idx, part_row, row_of, chain_status,
        chain_wcnt, chain_w, small;  // small: [0] blocks-done counter of the probe, [1] item count, [2] ticket, [3] exit counter
    DevBuf<uint4> items;
    void release() {
        tile_loc.release(); region_total.release(); part_idx.release(); part_row.release();
        row_of.release(); chain_status.release(); chain_wcnt.release();
        chain_w.release(); small.release(); items.release();
    }
};

struct rl_engine {
    int device = 0;
    cudaStream_t own_stream = nullptr, stream = nullptr;
    uint32_t cells = 1, log2P = 0, log2R = 0, row_bytes = 32;
    uint64_t capacity = 0;
    uint32_t max_batch = 0, max_counters = 0;
    uint8_t* d_rows = nullptr;

    // registry
    std::vector<HostLimit> limits;
    std::vector<HostGroup> groups;  // [0] unused
    std::map<std::pair<uint32_t, uint32_t>, std::vector<uint32_t>> groups_by_key;
    std::vector<std::vector<uint32_t>> ns_limits;  // registration order
    bool tables_dirty = true;
    bool any_multi_ns = false;
    uint32_t max_ns_limits = 0;
    uint32_t max_cells_used = 1;  // highest cell index + 1 over all row groups

    // device tables
    DevBuf<RlCellDesc> d_desc;
    DevBuf<RlLimitDev> d_limits;
    DevBuf<RlNsDev> d_ns;
    DevBuf<uint32_t> d_ns_limit_ids;
    DevBuf<uint32_t> d_group_ns;
    uint32_t limits_cap = 0, ns_cap = 0;

    // workspace
    DevBuf<uint32_t> d_tile_loc, d_region_total, d_part_idx, d_part_row, d_row_of, d_misc;  // misc: err, flags, scan_ctr, changed, ...
    DevBuf<RlAccess> d_acc;
    DevBuf<uint64_t> d_delta, d_now;
    DevBuf<uint32_t> d_fl_prev, d_fl_next;
    DevBuf<uint4> d_items;
    DevBuf<unsigned long long> d_kstats;
    DevBuf<uint4> d_trace;     // RL_FLAG_TRACE: event ring
    DevBuf<uint32_t> d_hot;    // [RL_HOT_SLOTS] hot rows + [RL_HOT_CAND] candidates + [1] candidate count
    bool hot_rows = false;     // RL_HOT=1 enables the hot-row partitions (k_hot); see DESIGN.md §3.4 for why it is opt-in
    DevBuf<uint32_t> d_misc2;  // [0] trace write position
    uint32_t trace_seq = 0;
    DevBuf<uint32_t> d_chain_status, d_chain_wcnt, d_chain_w;
    DevBuf<uint8_t*> d_log_row;
    DevBuf<ulonglong2> d_log_state;
    // staging for RL_MEM_HOST calls
    DevBuf<rl_record> d_in_recs;
    DevBuf<uint32_t> d_in_off;
    DevBuf<rl_counter> d_in_ctrs;
    DevBuf<uint64_t> d_in_delta, d_in_now;
    DevBuf<uint8_t> d_out_limited;
    DevBuf<uint32_t> d_out_first;
    DevBuf<uint64_t> d_out_rem, d_out_ttl;
    // bucket helper
    DevBuf<uint32_t> d_bucket;
    DevBuf<unsigned long long> d_bucket_counts;
    uint32_t* h_misc = nullptr;  // pinned mirror of d_misc

    rl_stats stats{};
    std::string last_error = "";
    // rl_profile_begin/end
    // RL_FLAG_PIPELINE
    bool pipeline = false;
    bool kernel_stats = false;  // RL_FLAG_KERNEL_STATS
    static constexpr int kSets = RL_SETS;  // workspace sets = calls in flight (probe | scan+scatter | replay)
    WorkSet wsx[kSets - 1];                // sets 1.. (set 0 = the engine's own members)
    cudaStream_t sq = nullptr;       // scan + scatter stream
    cudaStream_t sp = nullptr, sm = nullptr;  // partition / replay streams
    cudaEvent_t ev_in = nullptr, ev_probe[kSets] = {}, ev_part[kSets] = {}, ev_main[kSets] = {};  // ev_probe: replay done, before a post_main hook
    uint64_t pipe_seq = 0;
    bool pipe_pending = false;
    // RL_MEM_HOST_ASYNC: ring of device staging slots; copies overlap the kernels of other calls
    static constexpr int kRing = RL_RING;
    DevBuf<rl_record> ring_recs[kRing];
    DevBuf<uint8_t> ring_lim[kRing];
    DevBuf<uint32_t> ring_first[kRing];
    cudaEvent_t ev_slot[kRing] = {};  // slot's D2H done
    uint64_t ring_seq = 0;
    bool d2h_pending = false;
    int d2h_last = 0;
    uint32_t weak_slots = 0;           // RL_FLAG_DEBUG_WEAK_TAGS
    uint32_t chunk = 128;              // accesses per k_main chunk (128 or 256; RL_CHUNK overrides)
    uint32_t part_target = 128;        // accesses per partition aimed at (RL_PART_TARGET)
    uint32_t main_grid_cap = 148 * 16;  // k_main CTAs launched at most (SMs x 16)
    uint32_t heavy_mult = 2;           // regions > heavy_mult x average are chained (0 = never; RL_HEAVY_MULT)
    bool profiling = false;
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> prof_events;
    // rl_maint.cu: its per-engine state, and the per-namespace metrics hook (nullptr = off) called behind the replay
    // of a record call, on the stream that carries it
    void* ext = nullptr;
    void (*ext_free)(void*) = nullptr;
    rl_ns_hook_fn ns_hook = nullptr;
};

namespace {

enum { MISC_ERR = 0, MISC_FLAGS = 1, MISC_SCANCTR = 2, MISC_CHANGED = 3, MISC_NITEMS = 4, MISC_TICKET = 5, MISC_EXITCTR = 6, MISC_N = 8 };

int fail(rl_engine* e, int status, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (e) e->last_error = buf;
    return status;
}

int pipe_fence(rl_engine* e);

#define RL_CUDA(e, call)                                                                          \
    do {                                                                                          \
        cudaError_t _r = (call);                                                                  \
        if (_r != cudaSuccess)                                                                    \
            return fail((e), _r == cudaErrorMemoryAllocation ? RL_TRANSIENT : RL_FATAL,           \
                        "CUDA error %s at %s:%d (%s)", cudaGetErrorName(_r), __FILE__, __LINE__,  \
                        cudaGetErrorString(_r));                                                  \
    } while (0)

#define RL_LAUNCH_CHECK(e)                    \
    do {                                      \
        (e)->stats.kernel_launches++;         \
        RL_CUDA((e), cudaGetLastError());     \
    } while (0)

uint32_t ceil_div(uint64_t a, uint64_t b) { return (uint32_t)((a + b - 1) / b); }

uint32_t log2_ceil(uint64_t x) {
    uint32_t l = 0;
    while ((1ull << l) < x) l++;
    return l;
}

RlDev make_dev(rl_engine* e) {
    RlDev D;
    D.rows = e->d_rows;
    D.log2P = e->log2P;
    D.log2R = e->log2R;
    D.desc = e->d_desc.p;
    D.limits = e->d_limits.p;
    D.limits_cap = e->limits_cap;
    D.ns = e->d_ns.p;
    D.ns_cap = e->ns_cap;
    D.ns_limit_ids = e->d_ns_limit_ids.p;
    D.err = e->d_misc.p + MISC_ERR;
    D.flags = e->d_misc.p + MISC_FLAGS;
    D.kstats = e->kernel_stats ? e->d_kstats.p : nullptr;
    D.hot_rows = e->d_hot.p;
    D.hot_cand = e->d_hot.p + RL_HOT_SLOTS;
    D.hot_cand_n = e->d_hot.p + RL_HOT_SLOTS + RL_HOT_CAND;
    D.trace = e->d_trace.p;
    D.trace_pos = e->d_trace.p ? e->d_misc2.p : nullptr;
    D.seq = e->trace_seq;
    return D;
}

// Rebuild and upload the limit / group / namespace tables.
int upload_tables(rl_engine* e) {
    if (!e->tables_dirty) return RL_OK;
    const size_t ngroups = e->groups.size();
    std::vector<RlCellDesc> desc(ngroups * 8);
    std::vector<uint32_t> group_ns(ngroups, 0);
    for (auto& d : desc) {
        d.max_value = 0;
        d.window_us = 0;
        d.limit_id = RL_NONE_U32;
        d.qualified = 0;
    }
    e->max_cells_used = 1;
    for (size_t g = 1; g < ngroups; g++) {
        group_ns[g] = e->groups[g].ns;
        for (uint32_t c = 0; c < RL_MAX_CELLS; c++) {
            const uint32_t lid = e->groups[g].limit_of_cell[c];
            if (lid == RL_NONE_U32) continue;
            e->max_cells_used = std::max(e->max_cells_used, c + 1);
            const HostLimit& l = e->limits[lid];
            RlCellDesc& d = desc[g * 8 + c];
            d.max_value = l.max_value;
            d.window_us = l.window_us;
            d.limit_id = lid;
            d.qualified = l.qualified;
        }
    }
    std::vector<RlLimitDev> lim(std::max<size_t>(e->limits.size(), 1));
    for (size_t i = 0; i < lim.size(); i++) {
        lim[i].group = 0;
        lim[i].cell = 0;
        lim[i].ns_id = 0;
        lim[i].qualified = 0;
        if (i < e->limits.size() && e->limits[i].defined) {
            lim[i].group = e->limits[i].group;
            lim[i].cell = e->limits[i].cell;
            lim[i].ns_id = e->limits[i].ns;
            lim[i].qualified = e->limits[i].qualified;
        }
    }
    std::vector<RlNsDev> ns(std::max<size_t>(e->ns_limits.size(), 1));
    std::vector<uint32_t> ns_ids;
    e->any_multi_ns = false;
    e->max_ns_limits = 0;
    for (size_t n = 0; n < ns.size(); n++) {
        memset(&ns[n], 0, sizeof(RlNsDev));
        if (n >= e->ns_limits.size() || e->ns_limits[n].empty()) continue;
        const auto& L = e->ns_limits[n];
        ns[n].lim_off = (uint32_t)ns_ids.size();
        ns[n].lim_cnt = (uint32_t)L.size();
        e->max_ns_limits = std::max<uint32_t>(e->max_ns_limits, (uint32_t)L.size());
        bool single = L.size() <= RL_MAX_CELLS;
        for (uint32_t lid : L) {
            ns_ids.push_back(lid);
            if (e->limits[lid].group != e->limits[L[0]].group) single = false;
        }
        if (single) {
            ns[n].mode = 1;
            ns[n].group = e->limits[L[0]].group;
            ns[n].qualified_row = e->limits[L[0]].qualified;
            uint32_t cells = 0;
            for (size_t k = 0; k < L.size(); k++) cells |= e->limits[L[k]].cell << (4 * k);
            ns[n].cells = cells | ((uint32_t)L.size() << 28);
        } else {
            ns[n].mode = 2;
            e->any_multi_ns = true;
        }
    }
    if (ns_ids.empty()) ns_ids.push_back(0);
    RL_CUDA(e, e->d_desc.reserve(desc.size()));
    RL_CUDA(e, e->d_limits.reserve(lim.size()));
    RL_CUDA(e, e->d_ns.reserve(ns.size()));
    RL_CUDA(e, e->d_ns_limit_ids.reserve(ns_ids.size()));
    RL_CUDA(e, e->d_group_ns.reserve(group_ns.size()));
    // synchronous copies: the host vectors die at scope exit
    RL_CUDA(e, cudaStreamSynchronize(e->stream));
    RL_CUDA(e, cudaMemcpy(e->d_desc.p, desc.data(), desc.size() * sizeof(RlCellDesc), cudaMemcpyHostToDevice));
    RL_CUDA(e, cudaMemcpy(e->d_limits.p, lim.data(), lim.size() * sizeof(RlLimitDev), cudaMemcpyHostToDevice));
    RL_CUDA(e, cudaMemcpy(e->d_ns.p, ns.data(), ns.size() * sizeof(RlNsDev), cudaMemcpyHostToDevice));
    RL_CUDA(e, cudaMemcpy(e->d_ns_limit_ids.p, ns_ids.data(), ns_ids.size() * sizeof(uint32_t), cudaMemcpyHostToDevice));
    RL_CUDA(e, cudaMemcpy(e->d_group_ns.p, group_ns.data(), group_ns.size() * sizeof(uint32_t), cudaMemcpyHostToDevice));
    e->limits_cap = (uint32_t)lim.size();
    e->ns_cap = (uint32_t)ns.size();
    e->tables_dirty = false;
    return RL_OK;
}

// Translate the sticky device error (if any) into a status; clears it.
int check_device_error(rl_engine* e) {
    {
        int rf = pipe_fence(e);
        if (rf) return rf;
    }
    RL_CUDA(e, cudaMemcpyAsync(e->h_misc, e->d_misc.p, MISC_N * sizeof(uint32_t), cudaMemcpyDeviceToHost, e->stream));
    RL_CUDA(e, cudaStreamSynchronize(e->stream));
    const uint32_t code = e->h_misc[MISC_ERR];
    if (code == RL_DEV_OK) return RL_OK;
    RL_CUDA(e, cudaMemsetAsync(e->d_misc.p + MISC_ERR, 0, sizeof(uint32_t), e->stream));
    switch (code) {
        case RL_DEV_TABLE_FULL:
            return fail(e, RL_TRANSIENT, "counter table region full (capacity_rows=%llu): batch partially applied",
                        (unsigned long long)e->capacity);
        case RL_DEV_UNKNOWN_LIMIT:
            return fail(e, RL_FATAL, "request names a limit_id that was never registered with rl_limits_set");
        case RL_DEV_KEY_RANGE:
            return fail(e, RL_FATAL, "key_hi bits 32..55 must be zero (counter identity is a 96-bit digest)");
        case RL_DEV_TOO_MANY_COUNTERS:
            return fail(e, RL_FATAL, "a request has more than %d counters", RL_MAX_CTRS_PER_REQ);
        case RL_DEV_CLOCK:
            return fail(e, RL_FATAL, "now_us must be >= 1");
        case RL_DEV_EXCHANGE: {
            const uint32_t d = e->h_misc[7];
            RL_CUDA(e, cudaMemsetAsync(e->d_misc.p + 7, 0, sizeof(uint32_t), e->stream));
            const char* what = (d >> 28) == 1 ? "records of source rank" : (d >> 28) == 2 ? "verdicts of owner rank" : "inbox larger than max_batch, rank";
            return fail(e, RL_FATAL, "peer exchange failed at step %u: %s %u did not arrive within %.0f s (or a block fill was out of range)",
                        d & 0xFFFFFu, what, (d >> 20) & 0xFFu, (double)RL_XCHG_TIMEOUT_NS * 1e-9);
        }
        default:
            return fail(e, RL_FATAL, "device error code %u", code);
    }
}

// A resolve kernel (request -> accesses) found a request the engine cannot take (unknown limit, more than
// RL_MAX_COUNTERS_PER_REQUEST counters, key out of range): refuse the WHOLE call before anything touches the
// table, so that the caller can fix the batch and retry without double counting (ADVICE r1).
int check_resolve_error(rl_engine* e) {
    RL_CUDA(e, cudaMemcpyAsync(e->h_misc, e->d_misc.p, MISC_N * sizeof(uint32_t), cudaMemcpyDeviceToHost, e->stream));
    RL_CUDA(e, cudaStreamSynchronize(e->stream));
    if (e->h_misc[MISC_ERR] == RL_DEV_OK) return RL_OK;
    int r = check_device_error(e);
    if (r == RL_OK) r = RL_FATAL;
    e->last_error += " — the call was refused before the table was touched";
    return r;
}

struct Outs {
    uint8_t* limited = nullptr;
    uint32_t* first = nullptr;
    uint64_t* rem = nullptr;
    uint64_t* ttl = nullptr;
    const uint32_t* off = nullptr;
    uint32_t stride = 0;
};

RlBatch make_batch(rl_engine* e, uint32_t n_acc, uint32_t n_req, const Outs& o, int lc, int set = 0, uint32_t n_hint = 0,
                   bool hot_ok = true) {
    RlBatch B;
    B.nhot = (hot_ok && e->hot_rows) ? RL_HOT_SLOTS : 0;
    B.n_acc = n_acc;
    B.n_req = n_req;
    B.n_dev = nullptr;
    B.omap_prefix = nullptr;
    B.omap_n = 0;
    B.omap_stride = 0;
    B.tile_loc = e->d_tile_loc.p;
    B.region_total = e->d_region_total.p;
    B.part_idx = e->d_part_idx.p;
    B.row_of = e->d_row_of.p;
    B.part_row = e->d_part_row.p;
    B.scan_ctr = e->d_misc.p + MISC_SCANCTR;
    B.ticket = e->d_misc.p + MISC_TICKET;
    B.exit_ctr = e->d_misc.p + MISC_EXITCTR;
    uint32_t tile = ceil_div(n_acc, kMaxTiles);
    tile = std::max<uint32_t>(512, ((tile + 255) / 256) * 256);
    B.tile = tile;
    B.num_tiles = std::max<uint32_t>(1, ceil_div(n_acc, tile));
    // n_hint (sharded steps): n_acc is only the upper bound of a device-side count; partitions are sized for
    // the expected count, and the kernels derive the tile from the actual one (rl_tile_of)
    const uint32_t n_size = n_hint ? std::min(n_hint, n_acc) : n_acc;
    if (n_hint) B.num_tiles = std::min<uint32_t>(256, std::max<uint32_t>(1, ceil_div(n_acc, 256)));
    B.out_limited = o.limited;
    B.out_first_limited = o.first;
    B.out_remaining = o.rem;
    B.out_ttl = o.ttl;
    B.out_off = o.off;
    B.out_stride = o.stride;
    B.fl_prev = e->d_fl_prev.p;
    B.fl_next = e->d_fl_next.p;
    B.phase = RL_PHASE_COMMIT;
    B.load_counters = lc;
    B.items = e->d_items.p;
    B.n_items = e->d_misc.p + MISC_NITEMS;
    B.chain_status = e->d_chain_status.p;
    B.chain_wcnt = e->d_chain_wcnt.p;
    B.chain_w = e->d_chain_w.p;
    B.chunk = e->chunk;
    // a region is split into chained chunks only when it is far heavier than the average one
    // partition granularity: about one k_main chunk per partition, never finer than the table's regions
    {
        uint32_t want = std::max<uint32_t>(64, ceil_div(n_size, e->part_target));
        uint32_t lp = 0;
        while ((1u << (lp + 1)) <= want) lp++;
        lp = std::min<uint32_t>(lp, e->log2P);
        B.part_shift = e->log2P - lp;
        B.nparts = 1u << lp;
    }
    B.heavy_len = e->heavy_mult ? std::max<uint32_t>(2 * e->chunk, e->heavy_mult * ceil_div(n_size, B.nparts)) : 0xFFFFFFFFu;
    B.log_row = nullptr;
    B.log_state = nullptr;
    if (set >= 1) {
        WorkSet& w = e->wsx[set - 1];
        B.tile_loc = w.tile_loc.p;
        B.region_total = w.region_total.p;
        B.part_idx = w.part_idx.p;
        B.row_of = w.row_of.p;
        B.part_row = w.part_row.p;
        B.scan_ctr = w.small.p + 0;
        B.items = w.items.p;
        B.n_items = w.small.p + 1;
        B.ticket = w.small.p + 2;
        B.exit_ctr = w.small.p + 3;
        B.chain_status = w.chain_status.p;
        B.chain_wcnt = w.chain_wcnt.p;
        B.chain_w = w.chain_w.p;
    }
    return B;
}

template <int CELLS, class Src>
int launch_front_cells(rl_engine* e, const RlDev& D, const RlBatch& B, const Src& src, cudaStream_t st) {
    const uint32_t P1 = B.nparts + B.nhot + 1;
    const size_t smem = ((size_t)RL_PART_WARPS * P1 + P1 + 1) * sizeof(uint32_t);
    static int smem_limit[64] = {};  // per instantiation and device: raised as engines with more regions appear
    const int dv = e->device & 63;
    // (k_front also has ~8 KB of static shared memory: opt in well before the 48 KB default is reached)
    if (smem > 32 * 1024 && (int)smem > smem_limit[dv]) {
        const uint32_t maxP1 = (1u << e->log2P) + RL_HOT_SLOTS + 1;
        const int max_smem = (int)(((size_t)RL_PART_WARPS * maxP1 + maxP1 + 1) * sizeof(uint32_t));
        RL_CUDA(e, cudaFuncSetAttribute(k_front<CELLS, Src>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem));
        smem_limit[dv] = max_smem;
    }
    k_front<CELLS, Src><<<B.num_tiles, RL_PART_THREADS, smem, st>>>(D, B, src);
    RL_LAUNCH_CHECK(e);
    return RL_OK;
}

// probe + stable partition by table region (one launch)
template <class Src>
int launch_front(rl_engine* e, const RlDev& D, const RlBatch& B, const Src& src, cudaStream_t st = nullptr) {
    if (!st) st = e->stream;
    switch (e->cells) {
        case 1: return launch_front_cells<1, Src>(e, D, B, src, st);
        case 3: return launch_front_cells<3, Src>(e, D, B, src, st);
        default: return launch_front_cells<7, Src>(e, D, B, src, st);
    }
}

template <int GEO, int CELLS, class Src, int MODE, bool LC, int CH>
int launch_main_ch(rl_engine* e, const RlDev& D, const RlBatch& B, const Src& src, cudaStream_t st) {
    using Smem = RlMainSmem<CELLS, CH>;
    auto kern = k_main<GEO, CELLS, Src, MODE, CH, LC>;
    static bool attr_set[64] = {};  // per instantiation and device (function attributes are per device)
    static uint32_t resident[64] = {};
    const int dv = e->device & 63;
    if (!attr_set[dv]) {
        RL_CUDA(e, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        (int)rl_main_smem_bytes<CELLS, CH>(RL_MAX_TILES)));
        int per_sm = 0;
        RL_CUDA(e, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, CH, sizeof(Smem)));
        resident[dv] = (uint32_t)std::max(per_sm, 1) * (e->main_grid_cap / 16);  // CTAs that fit at once (one wave)
        attr_set[dv] = true;
    }
    // upper bound of the work-item count: one per partition + one per chunk of a heavy partition; CTAs take
    // items from a ticket, so a smaller grid only means that some CTAs take several
    // (capping the grid at one resident wave was measured: the CTAs that then take a second item make the kernel last
    // two chunk latencies — 29.5 instead of 23 us on C2)
    (void)resident;
    const uint32_t grid = std::min<uint32_t>(B.nparts + ceil_div(B.n_acc, CH), e->main_grid_cap);
    kern<<<grid, CH, rl_main_smem_bytes<CELLS, CH>(B.num_tiles), st>>>(D, B, src, e->weak_slots);
    return RL_OK;
}

template <int GEO, int CELLS, class Src, int MODE, bool LC>
int launch_main_cells(rl_engine* e, const RlDev& D, const RlBatch& B, const Src& src, cudaStream_t st) {
    if (B.nhot && B.phase == RL_PHASE_COMMIT) {
        // the hot rows' partitions: one CTA per hot slot (most exit at once), ahead of the cold partitions
        k_hot<GEO, CELLS, Src, MODE, LC><<<B.nhot, RL_HOT_THREADS, 0, st>>>(D, B, src);
        RL_LAUNCH_CHECK(e);
    }
    return e->chunk == 128 ? launch_main_ch<GEO, CELLS, Src, MODE, LC, 128>(e, D, B, src, st)
                           : launch_main_ch<GEO, CELLS, Src, MODE, LC, 256>(e, D, B, src, st);
}

template <class Src, int MODE>
int launch_main(rl_engine* e, const RlDev& D, const RlBatch& B, const Src& src, cudaStream_t st = nullptr) {
    if (!st) st = e->stream;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    if (e->profiling) {
        RL_CUDA(e, cudaEventCreate(&ev0));
        RL_CUDA(e, cudaEventCreate(&ev1));
        RL_CUDA(e, cudaEventRecord(ev0, st));
    }
    int r;
    const bool lc = (MODE == 0) && B.load_counters;
#define RL_MAIN_CASE(G, A) \
    r = lc ? launch_main_cells<G, A, Src, MODE, MODE == 0>(e, D, B, src, st) : launch_main_cells<G, A, Src, MODE, false>(e, D, B, src, st)
    if (e->cells == 1) RL_MAIN_CASE(1, 1);
    else if (e->cells == 3) RL_MAIN_CASE(3, 3);
    else if (e->max_cells_used <= 4) RL_MAIN_CASE(7, 4);  // 128-B rows of which at most 4 cells are in use
    else RL_MAIN_CASE(7, 7);
#undef RL_MAIN_CASE
    if (r) return r;
    RL_LAUNCH_CHECK(e);
    if (e->profiling) {
        RL_CUDA(e, cudaEventRecord(ev1, st));
        e->prof_events.emplace_back(ev0, ev1);
    }
    return RL_OK;
}

// Make the caller's stream wait for everything the pipeline still has in flight.
int pipe_fence(rl_engine* e) {
    if (!e->pipe_pending) return RL_OK;
    const int last = (int)((e->pipe_seq - 1) % rl_engine::kSets);
    RL_CUDA(e, cudaStreamWaitEvent(e->stream, e->ev_main[last], 0));
    if (e->d2h_pending) RL_CUDA(e, cudaStreamWaitEvent(e->stream, e->ev_slot[e->d2h_last], 0));
    e->d2h_pending = false;
    e->pipe_pending = false;
    return RL_OK;
}

// Runs partition + main for accesses that may contain multi-row requests (AccSrc).
// mode: 0 check_and_update, 2 update.
int run_acc_pipeline(rl_engine* e, uint32_t n_acc, uint32_t n_req, const uint64_t* d_delta, const uint64_t* d_now,
                     int mode, int lc, const Outs& o) {
    RlDev D = make_dev(e);
    // check_and_update in the general form may hold coupled (multi-row) requests, replayed in phases: partitions
    // stay sequential and no row gets a partition of its own
    RlBatch B = make_batch(e, n_acc, n_req, o, lc, 0, 0, mode != 0);
    if (mode == 0) B.heavy_len = 0xFFFFFFFFu;
    AccSrc src{e->d_acc.p, d_delta, d_now};
    int r = launch_front(e, D, B, src);
    if (r) return r;
    if (mode == 2) return launch_main<AccSrc, 2>(e, D, B, src);
    // does the batch contain coupled (multi-row) requests?
    RL_CUDA(e, cudaMemcpyAsync(e->h_misc, e->d_misc.p, MISC_N * sizeof(uint32_t), cudaMemcpyDeviceToHost, e->stream));
    RL_CUDA(e, cudaStreamSynchronize(e->stream));
    e->stats.fixed_point_rounds = 0;
    if (e->h_misc[MISC_FLAGS] & 1u) {
        RL_CUDA(e, cudaMemsetAsync(e->d_misc.p + MISC_FLAGS, 0, sizeof(uint32_t), e->stream));
        RL_CUDA(e, e->d_fl_prev.reserve(e->max_batch));
        RL_CUDA(e, e->d_fl_next.reserve(e->max_batch));
        B.fl_prev = e->d_fl_prev.p;
        B.fl_next = e->d_fl_next.p;
        RL_CUDA(e, cudaMemsetAsync(B.fl_prev, 0xFF, n_req * sizeof(uint32_t), e->stream));
        RL_CUDA(e, cudaMemsetAsync(B.fl_next, 0xFF, n_req * sizeof(uint32_t), e->stream));
        // undo log: original state of every row the batch touches
        const uint32_t buf_len = B.num_tiles * B.tile;  // positions of part_idx/part_row in use
        RL_CUDA(e, e->d_log_row.reserve(buf_len));
        RL_CUDA(e, e->d_log_state.reserve((size_t)buf_len * e->cells));
        B.log_row = e->d_log_row.p;
        B.log_state = e->d_log_state.p;
        RL_CUDA(e, cudaMemsetAsync(B.log_row, 0, (size_t)buf_len * sizeof(uint8_t*), e->stream));
        B.phase = RL_PHASE_SNAPSHOT;
        r = launch_main<AccSrc, 0>(e, D, B, src);
        if (r) return r;
        // Fixed-point iteration over the requests' first-limited positions (DESIGN.md §3.4):
        // each speculative round replays the batch from the committed table state.
        for (uint32_t round = 0;; round++) {
            if (round > n_req + 2) return fail(e, RL_FATAL, "fixed-point iteration did not converge");
            RL_CUDA(e, cudaMemsetAsync(e->d_misc.p + MISC_CHANGED, 0, sizeof(uint32_t), e->stream));
            B.phase = RL_PHASE_SPEC;
            r = launch_main<AccSrc, 0>(e, D, B, src);
            if (r) return r;
            switch (e->cells) {
                case 1: k_restore<1><<<ceil_div(buf_len, 256), 256, 0, e->stream>>>(buf_len, 1, B.log_row, B.log_state); break;
                case 3: k_restore<3><<<ceil_div(buf_len, 256), 256, 0, e->stream>>>(buf_len, 3, B.log_row, B.log_state); break;
                default: k_restore<7><<<ceil_div(buf_len, 256), 256, 0, e->stream>>>(buf_len, e->max_cells_used <= 4 ? 4 : 7, B.log_row, B.log_state); break;
            }
            RL_LAUNCH_CHECK(e);
            k_fl_step<<<ceil_div(n_req, 256), 256, 0, e->stream>>>(n_req, B.fl_prev, B.fl_next,
                                                                    e->d_misc.p + MISC_CHANGED);
            RL_LAUNCH_CHECK(e);
            RL_CUDA(e, cudaMemcpyAsync(e->h_misc, e->d_misc.p, MISC_N * sizeof(uint32_t), cudaMemcpyDeviceToHost,
                                       e->stream));
            RL_CUDA(e, cudaStreamSynchronize(e->stream));
            e->stats.fixed_point_rounds = round + 1;
            if (!(e->h_misc[MISC_CHANGED] & 1u)) break;
        }
    }
    B.phase = RL_PHASE_COMMIT;
    return launch_main<AccSrc, 0>(e, D, B, src);
}

// Hooks of the sharded step (rl_shard_*): the owner's inbox is a segmented record source whose size is
// only known on the device; `pre_probe` runs on the probe stream right before the probe (it waits for
// the peers' blocks), `post_main` on the replay stream right behind k_main (it returns the verdicts).
struct PipeHooks {
    RecordSrc src;
    const uint32_t* n_dev = nullptr;
    std::function<void(RlBatch&)> patch_batch;  // verdict routing of a sharded step
    std::function<int(cudaStream_t, int)> pre_probe, post_main;  // (stream, workspace set)
};

// compact_now != 0: d_recs points at n 16-byte rl_record16 stamped with that one clock reading
int run_record_pipeline(rl_engine* e, uint32_t n, const rl_record* d_recs, int mode, int lc, const Outs& o,
                        bool may_pipeline = false, const PipeHooks* hooks = nullptr, uint32_t n_hint = 0,
                        uint64_t compact_now = 0) {
    RlDev D = make_dev(e);
    if (hooks && !(may_pipeline && e->pipeline && !e->any_multi_ns))
        return fail(e, RL_FATAL, "sharded steps need RL_FLAG_PIPELINE and single-row namespaces");
    if (may_pipeline && e->pipeline && !e->any_multi_ns) {
        // Two-stage software pipeline over successive calls: the front (probe + partition, `sp`) of
        // batch s+1 (and s+2) overlaps the replay of batch s (`sm`).  The front only reads row headers
        // and claims empty rows; the replay only touches the cells of rows found by ITS front, and
        // replays stay in call order on `sm`, so the table sees the batches in order.
        const int k = (int)(e->pipe_seq % rl_engine::kSets);
        RlBatch B = make_batch(e, n, n, o, lc, k, n_hint);
        RecordSrc src{d_recs, nullptr, 0, 0, compact_now ? 1u : 0u, compact_now};
        if (hooks) {
            // the inbox is filled by the peers' kernels and handed over through step flags, not through
            // anything on the caller's stream
            src = hooks->src;
            B.n_dev = hooks->n_dev;
            if (hooks->patch_batch) hooks->patch_batch(B);
        } else {
            RL_CUDA(e, cudaEventRecord(e->ev_in, e->stream));  // inputs: whatever the caller enqueued so far
            RL_CUDA(e, cudaStreamWaitEvent(e->sp, e->ev_in, 0));
        }
        if (e->pipe_seq >= (uint64_t)rl_engine::kSets)
            RL_CUDA(e, cudaStreamWaitEvent(e->sp, e->ev_main[k], 0));  // workspace set k is free again
        int r = RL_OK;
        if (hooks && hooks->pre_probe && (r = hooks->pre_probe(e->sp, k))) return r;
        r = launch_front(e, D, B, src, e->sp);
        if (r) return r;
        RL_CUDA(e, cudaEventRecord(e->ev_part[k], e->sp));
        RL_CUDA(e, cudaStreamWaitEvent(e->sm, e->ev_part[k], 0));
        r = mode == 2 ? launch_main<RecordSrc, 2>(e, D, B, src, e->sm) : launch_main<RecordSrc, 0>(e, D, B, src, e->sm);
        if (r) return r;
        // per-namespace metrics (rl_ns_metrics_enable): one reduction kernel right behind the replay, same stream
        if (e->ns_hook && !hooks && mode == 0 && o.limited &&
            (r = e->ns_hook(e, e->sm, n, d_recs, compact_now ? 16 : 32, o.limited, o.first)))
            return r;
        if (hooks && hooks->post_main) {
            // the hook (a sharded step's verdict return) runs on its own stream: the replay of the next call does
            // not wait for it, only the reuse of this workspace set does
            RL_CUDA(e, cudaEventRecord(e->ev_probe[k], e->sm));
            RL_CUDA(e, cudaStreamWaitEvent(e->sq, e->ev_probe[k], 0));
            if ((r = hooks->post_main(e->sq, k))) return r;
            RL_CUDA(e, cudaEventRecord(e->ev_main[k], e->sq));
        } else {
            RL_CUDA(e, cudaEventRecord(e->ev_main[k], e->sm));
        }
        e->pipe_seq++;
        e->pipe_pending = true;
        return RL_OK;
    }
    {
        int r = pipe_fence(e);
        if (r) return r;
    }
    if (!e->any_multi_ns) {
        RlBatch B = make_batch(e, n, n, o, lc);
        RecordSrc src{d_recs, nullptr, 0, 0, compact_now ? 1u : 0u, compact_now};
        int r = launch_front(e, D, B, src);
        if (r) return r;
        r = mode == 2 ? launch_main<RecordSrc, 2>(e, D, B, src) : launch_main<RecordSrc, 0>(e, D, B, src);
        if (r == RL_OK && e->ns_hook && mode == 0 && o.limited)
            r = e->ns_hook(e, e->stream, n, d_recs, compact_now ? 16 : 32, o.limited, o.first);
        return r;
    }
    if (compact_now) return fail(e, RL_FATAL, "16-byte records need single-row namespaces (use the 32-byte form)");
    // some namespace spans several rows: materialise accesses (stride = max limits per ns)
    const uint32_t stride = std::max<uint32_t>(1, e->max_ns_limits);
    if (stride > RL_MAX_CTRS_PER_REQ)
        return fail(e, RL_FATAL, "a namespace has more than %d limits", RL_MAX_CTRS_PER_REQ);
    const uint64_t n_acc = (uint64_t)n * stride;
    if (n_acc > e->d_acc.n)
        return fail(e, RL_FATAL, "batch of %u records x %u limits exceeds max_counters=%u", n, stride, e->max_counters);
    RlResolveOut O{e->d_acc.p, e->d_delta.p, e->d_now.p, o.limited, o.first};
    k_resolve_records<<<ceil_div(n, 128), 128, 0, e->stream>>>(D, n, d_recs, stride, O, mode == 0);
    RL_LAUNCH_CHECK(e);
    {
        int r = check_resolve_error(e);
        if (r) return r;
    }
    int r = run_acc_pipeline(e, (uint32_t)n_acc, n, e->d_delta.p, e->d_now.p, mode, lc, o);
    if (r == RL_OK && e->ns_hook && mode == 0 && o.limited) r = e->ns_hook(e, e->stream, n, d_recs, 32, o.limited, o.first);
    return r;
}

int ensure_ready(rl_engine* e, uint64_t n, bool fence = true) {
    if (!e) return RL_FATAL;
    if (fence) {
        int rf = pipe_fence(e);
        if (rf) return rf;
    }
    if (n > e->max_batch) return fail(e, RL_FATAL, "batch of %llu exceeds max_batch=%u", (unsigned long long)n, e->max_batch);
    RL_CUDA(e, cudaSetDevice(e->device));
    if (e->tables_dirty && e->pipeline) {
        int r = pipe_fence(e);
        if (r) return r;
        RL_CUDA(e, cudaStreamSynchronize(e->sp));
        RL_CUDA(e, cudaStreamSynchronize(e->sq));
        RL_CUDA(e, cudaStreamSynchronize(e->sm));
    }
    return upload_tables(e);
}

// Force the (lazy) loading of the kernels a record-form check_and_update launches for this engine's geometry.
template <int GEO, int CELLS>
int preload_main(rl_engine* e) {
    cudaFuncAttributes fa;
    RL_CUDA(e, cudaFuncGetAttributes(&fa, k_hot<GEO, CELLS, RecordSrc, 0, false>));
    if (e->chunk == 128) {
        RL_CUDA(e, cudaFuncGetAttributes(&fa, k_main<GEO, CELLS, RecordSrc, 0, 128, false>));
        RL_CUDA(e, cudaFuncSetAttribute(k_main<GEO, CELLS, RecordSrc, 0, 128, false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        (int)rl_main_smem_bytes<CELLS, 128>(RL_MAX_TILES)));
    } else {
        RL_CUDA(e, cudaFuncGetAttributes(&fa, k_main<GEO, CELLS, RecordSrc, 0, 256, false>));
        RL_CUDA(e, cudaFuncSetAttribute(k_main<GEO, CELLS, RecordSrc, 0, 256, false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        (int)rl_main_smem_bytes<CELLS, 256>(RL_MAX_TILES)));
    }
    return RL_OK;
}
int preload_record_kernels(rl_engine* e) {
    cudaFuncAttributes fa;
    int r = upload_tables(e);  // max_cells_used selects the k_main instantiation
    if (r) return r;
    switch (e->cells) {
        case 1:
            RL_CUDA(e, cudaFuncGetAttributes(&fa, k_front<1, RecordSrc>));
            return preload_main<1, 1>(e);
        case 3:
            RL_CUDA(e, cudaFuncGetAttributes(&fa, k_front<3, RecordSrc>));
            return preload_main<3, 3>(e);
        default:
            RL_CUDA(e, cudaFuncGetAttributes(&fa, k_front<7, RecordSrc>));
            if ((r = preload_main<7, 4>(e))) return r;
            return preload_main<7, 7>(e);
    }
}

}  // namespace

// =======================================================================================
extern "C" {

uint32_t rl_owner_of(uint32_t ns_id, uint32_t world) {
    return world ? (uint32_t)(rl_mix64((uint64_t)ns_id + 0x51ed270b0a1fULL) % world) : 0;
}

const char* rl_last_error(rl_engine* e) { return e ? e->last_error.c_str() : "null engine"; }

int rl_engine_create(const rl_config* cfg, rl_engine** out) {
    if (!cfg || !out) return RL_FATAL;
    *out = nullptr;
    if (cfg->struct_size != sizeof(rl_config)) return RL_FATAL;
    if (cfg->cells_per_row != 1 && cfg->cells_per_row != 3 && cfg->cells_per_row != 7) return RL_FATAL;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0 || cfg->device >= ndev || cfg->device < 0) {
        // No CPU fallback exists: without a CUDA device the engine cannot be created.
        return RL_FATAL;
    }
    rl_engine* e = new rl_engine();
    *out = e;  // returned even on failure so the caller can read rl_last_error, then destroy
    e->device = cfg->device;
    RL_CUDA(e, cudaSetDevice(e->device));
    cudaDeviceProp prop;
    RL_CUDA(e, cudaGetDeviceProperties(&prop, e->device));
    if (prop.major < 10) return fail(e, RL_FATAL, "device sm_%d%d is not sm_100a", prop.major, prop.minor);
    e->main_grid_cap = (uint32_t)prop.multiProcessorCount * 16u;
    // The table is read one random 32-B sector (a row header, a cell) at a time: ask the L2 not to fetch the
    // neighbouring sector from HBM along with it (the default granularity is 64 B).  A hint; per device.
    if (const char* v = getenv("RL_L2_FETCH")) {
        if (atoi(v) > 0) cudaDeviceSetLimit(cudaLimitMaxL2FetchGranularity, (size_t)atoi(v));
    }
    RL_CUDA(e, cudaStreamCreateWithFlags(&e->own_stream, cudaStreamNonBlocking));
    e->stream = e->own_stream;
    e->cells = cfg->cells_per_row;
    e->row_bytes = 16 * (1 + e->cells);
    uint32_t lg = std::max<uint32_t>(log2_ceil(std::max<uint64_t>(cfg->capacity_rows, 64)), 6);
    e->capacity = 1ull << lg;
    uint32_t regions = cfg->regions;
    if (regions == 0) {
        // auto: >= 1024 rows per region, at most 1024 regions
        regions = (uint32_t)std::min<uint64_t>(1024, std::max<uint64_t>(1, e->capacity / 1024));
    }
    if (regions & (regions - 1)) return fail(e, RL_FATAL, "regions must be a power of two");
    if (regions > kMaxRegions || (uint64_t)regions * 16 > e->capacity)
        return fail(e, RL_FATAL, "regions=%u out of range for capacity %llu", regions, (unsigned long long)e->capacity);
    e->log2P = log2_ceil(regions);
    e->log2R = lg - e->log2P;
    if (e->log2R > 31) return fail(e, RL_FATAL, "rows per region exceeds 2^31; raise regions");
    if (lg > 31) return fail(e, RL_FATAL, "capacity_rows must not exceed 2^31");
    e->max_batch = std::max<uint32_t>(cfg->max_batch, 1);
    e->max_counters = cfg->max_counters ? cfg->max_counters : 4 * e->max_batch;
    e->max_counters = std::max(e->max_counters, e->max_batch);
    e->groups.resize(1);
    if (const char* v = getenv("RL_CHUNK")) e->chunk = (atoi(v) == 128) ? 128 : 256;
    if (const char* v = getenv("RL_HEAVY_MULT")) e->heavy_mult = (uint32_t)atoi(v);
    if (const char* v = getenv("RL_PART_TARGET")) e->part_target = std::max(16, atoi(v));
    if (cfg->flags & 1u) e->weak_slots = 1;  // RL_FLAG_DEBUG_WEAK_TAGS: four home slots in the grouping table

    const size_t bytes = (size_t)e->capacity * e->row_bytes;
    RL_CUDA(e, cudaMalloc((void**)&e->d_rows, bytes));
    RL_CUDA(e, cudaMemsetAsync(e->d_rows, 0, bytes, e->stream));

    const uint32_t P1 = (1u << e->log2P) + RL_HOT_SLOTS + 1;  // cold partitions + hot slots + the no-row bucket
    const size_t maxA = e->max_counters;
    const size_t bufA = maxA + maxA / 128 + 256 * 1024 + 1024;  // part_idx/part_row: every tile's slice is a whole tile
    RL_CUDA(e, e->d_tile_loc.reserve((size_t)(kMaxTiles + 1) * (P1 + 1)));
    RL_CUDA(e, e->d_region_total.reserve(P1 + 1));
    RL_CUDA(e, cudaMemsetAsync(e->d_region_total.p, 0, (P1 + 1) * sizeof(uint32_t), e->stream));
    RL_CUDA(e, e->d_part_idx.reserve(bufA));
    RL_CUDA(e, e->d_row_of.reserve(maxA));
    RL_CUDA(e, e->d_part_row.reserve(bufA));
    RL_CUDA(e, e->d_misc.reserve(MISC_N));
    RL_CUDA(e, cudaMemsetAsync(e->d_misc.p, 0, MISC_N * sizeof(uint32_t), e->stream));
    RL_CUDA(e, cudaMallocHost((void**)&e->h_misc, MISC_N * sizeof(uint32_t)));
    RL_CUDA(e, e->d_acc.reserve(maxA));
    RL_CUDA(e, e->d_kstats.reserve(32));
    RL_CUDA(e, cudaMemsetAsync(e->d_kstats.p, 0, 32 * sizeof(unsigned long long), e->stream));
    RL_CUDA(e, e->d_items.reserve((size_t)(1u << e->log2P) + maxA / 128 + 2));
    {
        const size_t max_items = (size_t)(1u << e->log2P) + maxA / 128 + 2;
        RL_CUDA(e, e->d_chain_status.reserve(max_items));
        RL_CUDA(e, e->d_chain_wcnt.reserve(max_items));
        RL_CUDA(e, e->d_chain_w.reserve(max_items * 256));
    }
    RL_CUDA(e, e->d_delta.reserve(e->max_batch));
    RL_CUDA(e, e->d_now.reserve(e->max_batch));
    e->kernel_stats = (cfg->flags & RL_FLAG_KERNEL_STATS) != 0;
    e->hot_rows = (cfg->flags & RL_FLAG_HOT_ROWS) != 0;
    if (const char* v = getenv("RL_HOT")) e->hot_rows = atoi(v) != 0;
    RL_CUDA(e, e->d_hot.reserve(RL_HOT_SLOTS + RL_HOT_CAND + 4));
    RL_CUDA(e, cudaMemsetAsync(e->d_hot.p, 0xFF, (RL_HOT_SLOTS + RL_HOT_CAND) * sizeof(uint32_t), e->stream));
    RL_CUDA(e, cudaMemsetAsync(e->d_hot.p + RL_HOT_SLOTS + RL_HOT_CAND, 0, 4 * sizeof(uint32_t), e->stream));
    RL_CUDA(e, e->d_misc2.reserve(4));
    RL_CUDA(e, cudaMemsetAsync(e->d_misc2.p, 0, 4 * sizeof(uint32_t), e->stream));
    if (cfg->flags & RL_FLAG_TRACE) {
        RL_CUDA(e, e->d_trace.reserve(RL_TRACE_CAP));
        RL_CUDA(e, cudaMemsetAsync(e->d_trace.p, 0, RL_TRACE_CAP * sizeof(uint4), e->stream));
    }
    if (cfg->flags & 2u) {  // RL_FLAG_PIPELINE
        e->pipeline = true;
        RL_CUDA(e, cudaStreamCreateWithFlags(&e->sp, cudaStreamNonBlocking));
        RL_CUDA(e, cudaStreamCreateWithFlags(&e->sm, cudaStreamNonBlocking));
        for (int k = 0; k < rl_engine::kRing; k++) RL_CUDA(e, cudaEventCreateWithFlags(&e->ev_slot[k], cudaEventDisableTiming));
        RL_CUDA(e, cudaEventCreateWithFlags(&e->ev_in, cudaEventDisableTiming));
        RL_CUDA(e, cudaStreamCreateWithFlags(&e->sq, cudaStreamNonBlocking));
        for (int k = 0; k < rl_engine::kSets; k++) {
            RL_CUDA(e, cudaEventCreateWithFlags(&e->ev_probe[k], cudaEventDisableTiming));
            RL_CUDA(e, cudaEventCreateWithFlags(&e->ev_part[k], cudaEventDisableTiming));
            RL_CUDA(e, cudaEventCreateWithFlags(&e->ev_main[k], cudaEventDisableTiming));
        }
        const size_t max_items = (size_t)(1u << e->log2P) + maxA / 128 + 2;
        for (int wi = 0; wi < rl_engine::kSets - 1; wi++) {
        WorkSet& w = e->wsx[wi];
        RL_CUDA(e, w.tile_loc.reserve((size_t)(kMaxTiles + 1) * (P1 + 1)));
        RL_CUDA(e, w.region_total.reserve(P1 + 1));
        RL_CUDA(e, cudaMemsetAsync(w.region_total.p, 0, (P1 + 1) * sizeof(uint32_t), e->stream));
        RL_CUDA(e, w.part_idx.reserve(bufA));
        RL_CUDA(e, w.part_row.reserve(bufA));
        RL_CUDA(e, w.row_of.reserve(maxA));
        RL_CUDA(e, w.items.reserve(max_items));
        RL_CUDA(e, w.chain_status.reserve(max_items));
        RL_CUDA(e, w.chain_wcnt.reserve(max_items));
        RL_CUDA(e, w.chain_w.reserve(max_items * 256));
        RL_CUDA(e, w.small.reserve(8));
        RL_CUDA(e, cudaMemsetAsync(w.small.p, 0, 8 * sizeof(uint32_t), e->stream));
        }
    }
    RL_CUDA(e, cudaStreamSynchronize(e->stream));
    e->stats.capacity_rows = e->capacity;
    e->stats.regions = 1u << e->log2P;
    e->stats.row_bytes = e->row_bytes;
    return RL_OK;
}

void rl_engine_destroy(rl_engine* e) {
    if (!e) return;
    cudaSetDevice(e->device);
    if (e->sp) cudaStreamSynchronize(e->sp);
    if (e->sm) cudaStreamSynchronize(e->sm);
    if (e->ext && e->ext_free) {
        if (e->stream) cudaStreamSynchronize(e->stream);
        e->ext_free(e->ext);
        e->ext = nullptr;
    }
    for (int k = 0; k < rl_engine::kRing; k++) {
        e->ring_recs[k].release();
        e->ring_lim[k].release();
        e->ring_first[k].release();
        if (e->ev_slot[k]) cudaEventDestroy(e->ev_slot[k]);
    }
    if (e->stream) cudaStreamSynchronize(e->stream);
    for (int k = 0; k < rl_engine::kSets - 1; k++) e->wsx[k].release();
    if (e->sq) cudaStreamSynchronize(e->sq);
    if (e->ev_in) cudaEventDestroy(e->ev_in);
    for (int k = 0; k < rl_engine::kSets; k++) {
        if (e->ev_probe[k]) cudaEventDestroy(e->ev_probe[k]);
        if (e->ev_part[k]) cudaEventDestroy(e->ev_part[k]);
        if (e->ev_main[k]) cudaEventDestroy(e->ev_main[k]);
    }
    if (e->sq) cudaStreamDestroy(e->sq);
    if (e->sp) cudaStreamDestroy(e->sp);
    if (e->sm) cudaStreamDestroy(e->sm);
    if (e->d_rows) cudaFree(e->d_rows);
    e->d_desc.release();
    e->d_limits.release();
    e->d_ns.release();
    e->d_ns_limit_ids.release();
    e->d_group_ns.release();
    e->d_tile_loc.release();
    e->d_region_total.release();
    e->d_part_idx.release();
    e->d_row_of.release();
    e->d_part_row.release();
    e->d_misc.release();
    e->d_acc.release();
    e->d_delta.release();
    e->d_now.release();
    e->d_fl_prev.release();
    e->d_fl_next.release();
    e->d_items.release();
    e->d_kstats.release();
    e->d_trace.release();
    e->d_hot.release();
    e->d_misc2.release();
    e->d_chain_status.release();
    e->d_chain_wcnt.release();
    e->d_chain_w.release();
    e->d_log_row.release();
    e->d_log_state.release();
    e->d_in_recs.release();
    e->d_in_off.release();
    e->d_in_ctrs.release();
    e->d_in_delta.release();
    e->d_in_now.release();
    e->d_out_limited.release();
    e->d_out_first.release();
    e->d_out_rem.release();
    e->d_out_ttl.release();
    e->d_bucket.release();
    e->d_bucket_counts.release();
    if (e->h_misc) cudaFreeHost(e->h_misc);
    if (e->own_stream) cudaStreamDestroy(e->own_stream);
    delete e;
}

int rl_engine_set_stream(rl_engine* e, void* cuda_stream) {
    if (!e) return RL_FATAL;
    RL_CUDA(e, cudaSetDevice(e->device));
    {
        int rf = pipe_fence(e);
        if (rf) return rf;
    }
    RL_CUDA(e, cudaStreamSynchronize(e->stream));
    e->stream = cuda_stream ? (cudaStream_t)cuda_stream : e->own_stream;
    return RL_OK;
}

void* rl_engine_stream(rl_engine* e) { return e ? (void*)e->stream : nullptr; }

int rl_sync(rl_engine* e) {
    if (!e) return RL_FATAL;
    RL_CUDA(e, cudaSetDevice(e->device));
    return check_device_error(e);
}

int rl_fence(rl_engine* e) {
    if (!e) return RL_FATAL;
    RL_CUDA(e, cudaSetDevice(e->device));
    return pipe_fence(e);
}

int rl_fence_call(rl_engine* e, uint32_t age) {
    if (!e) return RL_FATAL;
    RL_CUDA(e, cudaSetDevice(e->device));
    if (!e->pipeline || e->pipe_seq == 0) return RL_OK;
    if (age == 0) return pipe_fence(e);
    if (age >= (uint32_t)rl_engine::kSets) return fail(e, RL_FATAL, "rl_fence_call: age must be < %d", rl_engine::kSets);
    if (e->pipe_seq <= age) return RL_OK;
    // an earlier call: its replay event is still the one recorded for it
    RL_CUDA(e, cudaStreamWaitEvent(e->stream, e->ev_main[(e->pipe_seq - 1 - age) % rl_engine::kSets], 0));
    return RL_OK;
}

int rl_profile_begin(rl_engine* e) {
    if (!e) return RL_FATAL;
    e->profiling = true;
    return RL_OK;
}

int rl_profile_end(rl_engine* e, double* out_main_ms, uint64_t* out_main_launches) {
    if (!e) return RL_FATAL;
    RL_CUDA(e, cudaSetDevice(e->device));
    e->profiling = false;
    {
        int rf = pipe_fence(e);
        if (rf) return rf;
    }
    RL_CUDA(e, cudaStreamSynchronize(e->stream));
    double ms = 0;
    for (auto& pr : e->prof_events) {
        float t = 0;
        RL_CUDA(e, cudaEventElapsedTime(&t, pr.first, pr.second));
        ms += t;
        cudaEventDestroy(pr.first);
        cudaEventDestroy(pr.second);
    }
    if (out_main_ms) *out_main_ms = ms;
    if (out_main_launches) *out_main_launches = e->prof_events.size();
    e->prof_events.clear();
    return RL_OK;
}

int rl_trace_dump(rl_engine* e, uint32_t cap, uint32_t* out_ev, uint32_t* out_seq, uint64_t* out_ns, uint32_t* out_count) {
    if (!e || !out_count) return RL_FATAL;
    *out_count = 0;
    if (!e->d_trace.p) return RL_OK;
    RL_CUDA(e, cudaSetDevice(e->device));
    RL_CUDA(e, cudaDeviceSynchronize());
    uint32_t pos = 0;
    RL_CUDA(e, cudaMemcpy(&pos, e->d_misc2.p, sizeof pos, cudaMemcpyDeviceToHost));
    const uint32_t n = std::min<uint32_t>(pos, RL_TRACE_CAP);
    std::vector<uint4> ev(n);
    if (n) RL_CUDA(e, cudaMemcpy(ev.data(), e->d_trace.p, (size_t)n * sizeof(uint4), cudaMemcpyDeviceToHost));
    const uint32_t m = std::min(n, cap);
    for (uint32_t i = 0; i < m; i++) {
        out_ev[i] = ev[i].x;
        out_seq[i] = ev[i].y;
        out_ns[i] = ((uint64_t)ev[i].w << 32) | ev[i].z;
    }
    *out_count = m;
    RL_CUDA(e, cudaMemset(e->d_misc2.p, 0, sizeof(uint32_t)));
    return RL_OK;
}

int rl_get_stats(rl_engine* e, rl_stats* out) {
    if (!e || !out) return RL_FATAL;
    RL_CUDA(e, cudaSetDevice(e->device));
    {
        int rf = pipe_fence(e);
        if (rf) return rf;
    }
    unsigned long long ks[32];
    RL_CUDA(e, cudaMemcpyAsync(ks, e->d_kstats.p, sizeof ks, cudaMemcpyDeviceToHost, e->stream));
    RL_CUDA(e, cudaStreamSynchronize(e->stream));
    e->stats.chunks = ks[0];
    e->stats.replay_rounds = ks[1];
    e->stats.chained_chunks = ks[2];
    e->stats.ordered_chunks = ks[3];
    for (int i = 0; i < 6; i++) e->stats.phase_cycles[i] = ks[8 + i];
    e->stats.phase_cycles[1] = ks[16];  // slot 1 (unused by k_main): ns spent in the front's last-block tail
    {
        uint32_t hot[RL_HOT_SLOTS];
        RL_CUDA(e, cudaMemcpyAsync(hot, e->d_hot.p, sizeof hot, cudaMemcpyDeviceToHost, e->stream));
        RL_CUDA(e, cudaStreamSynchronize(e->stream));
        e->stats.hot_rows = 0;
        for (uint32_t h : hot) e->stats.hot_rows += (h != 0xFFFFFFFFu);
    }
    *out = e->stats;
    return RL_OK;
}

int rl_limits_set(rl_engine* e, const rl_limit_desc* limits, uint32_t n) {
    if (!e || (!limits && n)) return RL_FATAL;
    for (uint32_t i = 0; i < n; i++) {
        const rl_limit_desc& d = limits[i];
        if (d.limit_id == RL_NONE_U32) return fail(e, RL_FATAL, "limit_id 0xFFFFFFFF is reserved");
        if (d.limit_id > (1u << 26) || d.ns_id > (1u << 26))
            return fail(e, RL_FATAL, "limit_id / ns_id must be dense (<= 2^26)");
        const uint32_t q = d.qualified ? 1 : 0;
        const uint32_t varset = q ? d.varset_id : 0;
        if (q && d.varset_id == 0) return fail(e, RL_FATAL, "qualified limits need varset_id != 0");
        if (d.limit_id >= e->limits.size()) e->limits.resize(d.limit_id + 1);
        HostLimit& l = e->limits[d.limit_id];
        if (l.defined) {
            // Storage::update_limit (storage/mod.rs:67-83): identity fixed, max_value swapped
            if (l.ns != d.ns_id || l.window_us != d.window_us || l.qualified != q || l.varset != varset)
                return fail(e, RL_FATAL, "limit %u: namespace/window/variables are part of a limit's identity", d.limit_id);
            if (l.max_value != d.max_value) {
                l.max_value = d.max_value;
                e->tables_dirty = true;
            }
            if (!q) l.simple_present = true;  // add_counter: entry().or_default() (in_memory.rs:38-44)
            continue;
        }
        // pick a row group with a free cell
        auto& glist = e->groups_by_key[{d.ns_id, varset}];
        uint32_t g = 0, c = 0;
        for (uint32_t cand : glist) {
            for (uint32_t k = 0; k < e->cells; k++)
                if (e->groups[cand].limit_of_cell[k] == RL_NONE_U32) {
                    g = cand;
                    c = k;
                    break;
                }
            if (g) break;
        }
        if (!g) {
            if (e->groups.size() >= 0xFFFFFFF0u) return fail(e, RL_FATAL, "too many row groups");
            g = (uint32_t)e->groups.size();
            e->groups.emplace_back();
            e->groups[g].ns = d.ns_id;
            e->groups[g].varset = varset;
            e->groups[g].qualified = q;
            glist.push_back(g);
            c = 0;
        }
        e->groups[g].limit_of_cell[c] = d.limit_id;
        l.defined = true;
        l.ns = d.ns_id;
        l.varset = varset;
        l.qualified = q;
        l.max_value = d.max_value;
        l.window_us = d.window_us;
        l.group = g;
        l.cell = c;
        l.simple_present = !q;
        if (d.ns_id >= e->ns_limits.size()) e->ns_limits.resize(d.ns_id + 1);
        e->ns_limits[d.ns_id].push_back(d.limit_id);
        e->tables_dirty = true;
    }
    return RL_OK;
}

static int reset_selected(rl_engine* e, const std::vector<uint8_t>& sel) {
    int r = pipe_fence(e);
    if (r) return r;
    r = upload_tables(e);
    if (r) return r;
    DevBuf<uint8_t> d_sel;
    RL_CUDA(e, d_sel.reserve(std::max<size_t>(sel.size(), 1)));
    RL_CUDA(e, cudaMemcpyAsync(d_sel.p, sel.data(), sel.size(), cudaMemcpyHostToDevice, e->stream));
    RlDev D = make_dev(e);
    const uint32_t blocks = ceil_div(e->capacity, 256);
    switch (e->cells) {
        case 1: k_reset<1><<<blocks, 256, 0, e->stream>>>(D, e->capacity, 0, 0, d_sel.p, nullptr); break;
        case 3: k_reset<3><<<blocks, 256, 0, e->stream>>>(D, e->capacity, 0, 0, d_sel.p, nullptr); break;
        default: k_reset<7><<<blocks, 256, 0, e->stream>>>(D, e->capacity, 0, 0, d_sel.p, nullptr); break;
    }
    RL_LAUNCH_CHECK(e);
    RL_CUDA(e, cudaStreamSynchronize(e->stream));
    d_sel.release();
    return RL_OK;
}

int rl_delete_counters(rl_engine* e, const uint32_t* limit_ids, uint32_t n) {
    if (!e) return RL_FATAL;
    RL_CUDA(e, cudaSetDevice(e->device));
    std::vector<uint8_t> sel(std::max<size_t>(e->limits.size(), 1), 0);
    bool any = false;
    for (uint32_t i = 0; i < n; i++) {
        const uint32_t id = limit_ids[i];
        if (id >= e->limits.size() || !e->limits[id].defined) continue;
        sel[id] = 1;
        any = true;
        if (!e->limits[id].qualified) e->limits[id].simple_present = false;  // in_memory.rs:242-243
    }
    return any ? reset_selected(e, sel) : RL_OK;
}

int rl_limits_delete(rl_engine* e, const uint32_t* limit_ids, uint32_t n) {
    if (!e) return RL_FATAL;
    int r = rl_delete_counters(e, limit_ids, n);  // storage/mod.rs:104 — counters first
    if (r) return r;
    for (uint32_t i = 0; i < n; i++) {
        const uint32_t id = limit_ids[i];
        if (id >= e->limits.size() || !e->limits[id].defined) continue;
        HostLimit& l = e->limits[id];
        e->groups[l.group].limit_of_cell[l.cell] = RL_NONE_U32;
        auto& v = e->ns_limits[l.ns];
        v.erase(std::remove(v.begin(), v.end(), id), v.end());
        l = HostLimit();
        e->tables_dirty = true;
    }
    return RL_OK;
}

int rl_clear(rl_engine* e) {
    if (!e) return RL_FATAL;
    RL_CUDA(e, cudaSetDevice(e->device));
    // in_memory.rs:197-201 — only simple_limits is cleared
    std::vector<uint8_t> sel(std::max<size_t>(e->limits.size(), 1), 0);
    bool any = false;
    for (size_t id = 0; id < e->limits.size(); id++)
        if (e->limits[id].defined && !e->limits[id].qualified) {
            sel[id] = 1;
            any = true;
            e->limits[id].simple_present = false;
        }
    return any ? reset_selected(e, sel) : RL_OK;
}

int rl_sweep(rl_engine* e, uint64_t now_us, uint64_t* out_invalidated) {
    if (!e) return RL_FATAL;
    RL_CUDA(e, cudaSetDevice(e->device));
    int r = pipe_fence(e);
    if (r) return r;
    r = upload_tables(e);
    if (r) return r;
    DevBuf<unsigned long long> d_cnt;
    RL_CUDA(e, d_cnt.reserve(1));
    RL_CUDA(e, cudaMemsetAsync(d_cnt.p, 0, sizeof(unsigned long long), e->stream));
    RlDev D = make_dev(e);
    const uint32_t blocks = ceil_div(e->capacity, 256);
    switch (e->cells) {
        case 1: k_reset<1><<<blocks, 256, 0, e->stream>>>(D, e->capacity, 1, now_us, nullptr, d_cnt.p); break;
        case 3: k_reset<3><<<blocks, 256, 0, e->stream>>>(D, e->capacity, 1, now_us, nullptr, d_cnt.p); break;
        default: k_reset<7><<<blocks, 256, 0, e->stream>>>(D, e->capacity, 1, now_us, nullptr, d_cnt.p); break;
    }
    RL_LAUNCH_CHECK(e);
    unsigned long long cnt = 0;
    RL_CUDA(e, cudaMemcpyAsync(&cnt, d_cnt.p, sizeof cnt, cudaMemcpyDeviceToHost, e->stream));
    RL_CUDA(e, cudaStreamSynchronize(e->stream));
    d_cnt.release();
    if (out_invalidated) *out_invalidated = cnt;
    return RL_OK;
}

// shared by rl_dump_table (mode 0) and rl_get_counters (mode 1)
static int scan_table(rl_engine* e, int mode, uint64_t now_us, const std::vector<uint8_t>& ns_sel, uint64_t cap,
                      uint32_t* out_limit_id, uint64_t* out_key_lo, uint64_t* out_key_hi, uint64_t* out_a,
                      uint64_t* out_b, uint64_t* out_count) {
    int r = pipe_fence(e);
    if (r) return r;
    r = upload_tables(e);
    if (r) return r;
    // device capacity: every live cell could match; bound by cap + unqualified fix-ups
    const uint64_t dcap = std::max<uint64_t>(cap, 1);
    DevBuf<uint32_t> d_lid;
    DevBuf<uint64_t> d_lo, d_hi, d_a, d_b;
    DevBuf<unsigned long long> d_cnt;
    DevBuf<uint8_t> d_sel;
    RL_CUDA(e, d_lid.reserve(dcap));
    RL_CUDA(e, d_lo.reserve(dcap));
    RL_CUDA(e, d_hi.reserve(dcap));
    RL_CUDA(e, d_a.reserve(dcap));
    RL_CUDA(e, d_b.reserve(dcap));
    RL_CUDA(e, d_cnt.reserve(1));
    RL_CUDA(e, d_sel.reserve(std::max<size_t>(ns_sel.size(), 1)));
    RL_CUDA(e, cudaMemsetAsync(d_cnt.p, 0, sizeof(unsigned long long), e->stream));
    if (!ns_sel.empty())
        RL_CUDA(e, cudaMemcpyAsync(d_sel.p, ns_sel.data(), ns_sel.size(), cudaMemcpyHostToDevice, e->stream));
    RlDev D = make_dev(e);
    RlScanOut O{d_lid.p, d_lo.p, d_hi.p, d_a.p, d_b.p, d_cnt.p, dcap};
    const uint32_t blocks = ceil_div(e->capacity, 256);
    switch (e->cells) {
        case 1: k_scan<1><<<blocks, 256, 0, e->stream>>>(D, e->capacity, mode, now_us, d_sel.p, e->d_group_ns.p, O); break;
        case 3: k_scan<3><<<blocks, 256, 0, e->stream>>>(D, e->capacity, mode, now_us, d_sel.p, e->d_group_ns.p, O); break;
        default: k_scan<7><<<blocks, 256, 0, e->stream>>>(D, e->capacity, mode, now_us, d_sel.p, e->d_group_ns.p, O); break;
    }
    RL_LAUNCH_CHECK(e);
    unsigned long long cnt = 0;
    RL_CUDA(e, cudaMemcpyAsync(&cnt, d_cnt.p, sizeof cnt, cudaMemcpyDeviceToHost, e->stream));
    RL_CUDA(e, cudaStreamSynchronize(e->stream));
    const uint64_t got = std::min<uint64_t>(cnt, dcap);
    std::vector<uint32_t> lid(got);
    std::vector<uint64_t> lo(got), hi(got), a(got), b(got);
    if (got) {
        RL_CUDA(e, cudaMemcpy(lid.data(), d_lid.p, got * 4, cudaMemcpyDeviceToHost));
        RL_CUDA(e, cudaMemcpy(lo.data(), d_lo.p, got * 8, cudaMemcpyDeviceToHost));
        RL_CUDA(e, cudaMemcpy(hi.data(), d_hi.p, got * 8, cudaMemcpyDeviceToHost));
        RL_CUDA(e, cudaMemcpy(a.data(), d_a.p, got * 8, cudaMemcpyDeviceToHost));
        RL_CUDA(e, cudaMemcpy(b.data(), d_b.p, got * 8, cudaMemcpyDeviceToHost));
    }
    d_lid.release();
    d_lo.release();
    d_hi.release();
    d_a.release();
    d_b.release();
    d_cnt.release();
    d_sel.release();
    // host fix-up of unqualified counters: present iff simple_present (in_memory.rs:14,38-44)
    uint64_t w = 0, total = 0;
    std::vector<uint8_t> seen(e->limits.size() + 1, 0);
    auto emit = [&](uint32_t l, uint64_t klo, uint64_t khi, uint64_t va, uint64_t vb) {
        if (w < cap) {
            out_limit_id[w] = l;
            out_key_lo[w] = klo;
            out_key_hi[w] = khi;
            out_a[w] = va;
            out_b[w] = vb;
            w++;
        }
        total++;
    };
    for (uint64_t i = 0; i < got; i++) {
        const uint32_t l = lid[i];
        if (l < e->limits.size() && e->limits[l].defined && !e->limits[l].qualified) {
            if (!e->limits[l].simple_present) continue;
            seen[l] = 1;
        }
        emit(l, lo[i], hi[i], a[i], b[i]);
    }
    if (mode == 0) {
        // unqualified counters whose row was never touched are still present as (0, EPOCH)
        for (size_t l = 0; l < e->limits.size(); l++)
            if (e->limits[l].defined && !e->limits[l].qualified && e->limits[l].simple_present && !seen[l])
                emit((uint32_t)l, 0, 0, 0, 0);
    }
    total += (cnt > dcap) ? (cnt - dcap) : 0;
    if (out_count) *out_count = total;
    return RL_OK;
}

int rl_dump_table(rl_engine* e, uint64_t cap, uint32_t* out_limit_id, uint64_t* out_key_lo, uint64_t* out_key_hi,
                  uint64_t* out_value, uint64_t* out_expiry_us, uint64_t* out_count) {
    if (!e) return RL_FATAL;
    RL_CUDA(e, cudaSetDevice(e->device));
    std::vector<uint8_t> none;
    return scan_table(e, 0, 0, none, cap, out_limit_id, out_key_lo, out_key_hi, out_value, out_expiry_us, out_count);
}

int rl_get_counters(rl_engine* e, const uint32_t* limit_ids, uint32_t n, uint64_t now_us, uint64_t cap,
                    uint32_t* out_limit_id, uint64_t* out_key_lo, uint64_t* out_key_hi, uint64_t* out_remaining,
                    uint64_t* out_ttl_us, uint64_t* out_count) {
    if (!e) return RL_FATAL;
    RL_CUDA(e, cudaSetDevice(e->device));
    // in_memory.rs:161-171: counters_in_namespace(limit.namespace()) for every given limit
    std::vector<uint8_t> ns_sel(std::max<size_t>(e->ns_limits.size(), 1), 0);
    for (uint32_t i = 0; i < n; i++) {
        const uint32_t id = limit_ids[i];
        if (id < e->limits.size() && e->limits[id].defined) ns_sel[e->limits[id].ns] = 1;
    }
    return scan_table(e, 1, now_us, ns_sel, cap, out_limit_id, out_key_lo, out_key_hi, out_remaining, out_ttl_us,
                      out_count);
}

// ---------------------------------------------------------------------------------------
static int stage_outs(rl_engine* e, uint64_t n, uint64_t n_ctr_out, bool want_first, bool want_lc, Outs& dev) {
    RL_CUDA(e, e->d_out_limited.reserve(e->max_batch));
    dev.limited = e->d_out_limited.p;
    if (want_first) {
        RL_CUDA(e, e->d_out_first.reserve(e->max_batch));
        dev.first = e->d_out_first.p;
    }
    if (want_lc) {
        RL_CUDA(e, e->d_out_rem.reserve(std::max<uint64_t>(n_ctr_out, e->max_counters)));
        RL_CUDA(e, e->d_out_ttl.reserve(std::max<uint64_t>(n_ctr_out, e->max_counters)));
        dev.rem = e->d_out_rem.p;
        dev.ttl = e->d_out_ttl.p;
    }
    (void)n;
    return RL_OK;
}

int rl_check_and_update_records(rl_engine* e, uint64_t n, const rl_record* recs, int load_counters, int mem,
                                uint8_t* out_limited, uint32_t* out_first_limited, uint64_t* out_remaining,
                                uint64_t* out_ttl_us, uint32_t out_stride) {
    const bool host_async = (mem == RL_MEM_HOST_ASYNC) && e && e->pipeline && !e->any_multi_ns &&
                            !(load_counters && (out_remaining || out_ttl_us));
    if (mem == RL_MEM_HOST_ASYNC && !host_async) mem = RL_MEM_HOST;  // not available: plain synchronous call
    int r = ensure_ready(e, n, mem == RL_MEM_HOST);
    if (r) return r;
    if (n == 0) return RL_OK;
    if (!recs || !out_limited) return fail(e, RL_FATAL, "null recs/out_limited");
    const bool lc = load_counters && (out_remaining || out_ttl_us);
    if (lc && out_stride < e->max_ns_limits)
        return fail(e, RL_FATAL, "out_stride %u < limits per namespace %u", out_stride, e->max_ns_limits);
    e->stats.batches++;
    e->stats.requests += n;
    e->trace_seq = (uint32_t)e->stats.batches;
    if (mem == RL_MEM_DEVICE) {
        Outs o;
        o.limited = out_limited;
        o.first = out_first_limited;
        o.rem = lc ? out_remaining : nullptr;
        o.ttl = lc ? out_ttl_us : nullptr;
        o.stride = out_stride;
        return run_record_pipeline(e, (uint32_t)n, recs, 0, load_counters ? 1 : 0, o, true);
    }
    if (host_async) {
        // H2D on the caller's stream (which carries nothing else of ours), kernels on the pipeline
        // streams, D2H behind the replay: the copies of one call overlap the kernels of its neighbours.
        const int slot = (int)(e->ring_seq % rl_engine::kRing);
        RL_CUDA(e, e->ring_recs[slot].reserve(e->max_batch));
        RL_CUDA(e, e->ring_lim[slot].reserve(e->max_batch));
        if (out_first_limited) RL_CUDA(e, e->ring_first[slot].reserve(e->max_batch));
        if (e->ring_seq >= (uint64_t)rl_engine::kRing)
            RL_CUDA(e, cudaStreamWaitEvent(e->stream, e->ev_slot[slot], 0));  // slot drained (its D2H done)
        RL_CUDA(e, cudaMemcpyAsync(e->ring_recs[slot].p, recs, n * sizeof(rl_record), cudaMemcpyHostToDevice, e->stream));
        Outs o;
        o.limited = e->ring_lim[slot].p;
        o.first = out_first_limited ? e->ring_first[slot].p : nullptr;
        o.stride = out_stride;
        if ((r = run_record_pipeline(e, (uint32_t)n, e->ring_recs[slot].p, 0, load_counters ? 1 : 0, o, true))) return r;
        // The verdicts leave on the replay stream itself, right behind their k_main.  A dedicated copy
        // stream parked on "replay done" looked cleaner, but streams share hardware queues: whenever
        // it landed on the queue of the stream carrying the next H2D, that copy waited for the replay
        // too and the whole pipeline serialised (e2e 0.4 instead of 1.1 G decisions/s, one run in three).
        cudaStream_t sd = e->sm;
        RL_CUDA(e, cudaMemcpyAsync(out_limited, o.limited, n, cudaMemcpyDeviceToHost, sd));
        if (out_first_limited)
            RL_CUDA(e, cudaMemcpyAsync(out_first_limited, o.first, n * 4, cudaMemcpyDeviceToHost, sd));
        RL_CUDA(e, cudaEventRecord(e->ev_slot[slot], sd));
        e->d2h_pending = true;
        e->d2h_last = slot;
        e->ring_seq++;
        return RL_OK;
    }
    RL_CUDA(e, e->d_in_recs.reserve(e->max_batch));
    RL_CUDA(e, cudaMemcpyAsync(e->d_in_recs.p, recs, n * sizeof(rl_record), cudaMemcpyHostToDevice, e->stream));
    Outs o;
    const uint64_t nout = lc ? n * out_stride : 0;
    if ((r = stage_outs(e, n, nout, out_first_limited != nullptr, lc, o))) return r;
    o.stride = out_stride;
    if (lc) {
        // slots of limits a namespace does not have stay 0
        RL_CUDA(e, cudaMemsetAsync(o.rem, 0, nout * 8, e->stream));
        RL_CUDA(e, cudaMemsetAsync(o.ttl, 0, nout * 8, e->stream));
    }
    if ((r = run_record_pipeline(e, (uint32_t)n, e->d_in_recs.p, 0, load_counters ? 1 : 0, o))) return r;
    RL_CUDA(e, cudaMemcpyAsync(out_limited, o.limited, n, cudaMemcpyDeviceToHost, e->stream));
    if (out_first_limited)
        RL_CUDA(e, cudaMemcpyAsync(out_first_limited, o.first, n * 4, cudaMemcpyDeviceToHost, e->stream));
    if (lc && out_remaining) RL_CUDA(e, cudaMemcpyAsync(out_remaining, o.rem, nout * 8, cudaMemcpyDeviceToHost, e->stream));
    if (lc && out_ttl_us) RL_CUDA(e, cudaMemcpyAsync(out_ttl_us, o.ttl, nout * 8, cudaMemcpyDeviceToHost, e->stream));
    return check_device_error(e);
}

int rl_check_and_update_compact(rl_engine* e, uint64_t n, const rl_record16* recs, uint64_t now_us, int mem,
                                uint8_t* out_limited, uint32_t* out_first_limited) {
    const bool host_async = (mem == RL_MEM_HOST_ASYNC) && e && e->pipeline && !e->any_multi_ns;
    if (mem == RL_MEM_HOST_ASYNC && !host_async) mem = RL_MEM_HOST;
    int r = ensure_ready(e, n, mem == RL_MEM_HOST);
    if (r) return r;
    if (n == 0) return RL_OK;
    if (!recs || !out_limited) return fail(e, RL_FATAL, "null recs/out_limited");
    if (now_us == 0) return fail(e, RL_FATAL, "now_us must be >= 1");
    e->stats.batches++;
    e->stats.requests += n;
    e->trace_seq = (uint32_t)e->stats.batches;
    const rl_record* as32 = reinterpret_cast<const rl_record*>(recs);  // RecordSrc::compact reads 16-byte strides
    if (mem == RL_MEM_DEVICE) {
        Outs o;
        o.limited = out_limited;
        o.first = out_first_limited;
        return run_record_pipeline(e, (uint32_t)n, as32, 0, 0, o, true, nullptr, 0, now_us);
    }
    if (host_async) {
        const int slot = (int)(e->ring_seq % rl_engine::kRing);
        RL_CUDA(e, e->ring_recs[slot].reserve(e->max_batch));
        RL_CUDA(e, e->ring_lim[slot].reserve(e->max_batch));
        if (out_first_limited) RL_CUDA(e, e->ring_first[slot].reserve(e->max_batch));
        if (e->ring_seq >= (uint64_t)rl_engine::kRing)
            RL_CUDA(e, cudaStreamWaitEvent(e->stream, e->ev_slot[slot], 0));
        RL_CUDA(e, cudaMemcpyAsync(e->ring_recs[slot].p, recs, n * sizeof(rl_record16), cudaMemcpyHostToDevice, e->stream));
        Outs o;
        o.limited = e->ring_lim[slot].p;
        o.first = out_first_limited ? e->ring_first[slot].p : nullptr;
        if ((r = run_record_pipeline(e, (uint32_t)n, e->ring_recs[slot].p, 0, 0, o, true, nullptr, 0, now_us))) return r;
        cudaStream_t sd = e->sm;
        RL_CUDA(e, cudaMemcpyAsync(out_limited, o.limited, n, cudaMemcpyDeviceToHost, sd));
        if (out_first_limited)
            RL_CUDA(e, cudaMemcpyAsync(out_first_limited, o.first, n * 4, cudaMemcpyDeviceToHost, sd));
        RL_CUDA(e, cudaEventRecord(e->ev_slot[slot], sd));
        e->d2h_pending = true;
        e->d2h_last = slot;
        e->ring_seq++;
        return RL_OK;
    }
    RL_CUDA(e, e->d_in_recs.reserve(e->max_batch));
    RL_CUDA(e, cudaMemcpyAsync(e->d_in_recs.p, recs, n * sizeof(rl_record16), cudaMemcpyHostToDevice, e->stream));
    Outs o;
    if ((r = stage_outs(e, n, 0, out_first_limited != nullptr, false, o))) return r;
    if ((r = run_record_pipeline(e, (uint32_t)n, e->d_in_recs.p, 0, 0, o, false, nullptr, 0, now_us))) return r;
    RL_CUDA(e, cudaMemcpyAsync(out_limited, o.limited, n, cudaMemcpyDeviceToHost, e->stream));
    if (out_first_limited)
        RL_CUDA(e, cudaMemcpyAsync(out_first_limited, o.first, n * 4, cudaMemcpyDeviceToHost, e->stream));
    return check_device_error(e);
}

// Brings a CSR batch onto the device (or aliases it) and returns the total counter count.
struct CsrDev {
    const uint32_t* off = nullptr;
    const rl_counter* ctrs = nullptr;
    const uint64_t* delta = nullptr;
    const uint64_t* now = nullptr;
    uint64_t total = 0;
};

static int stage_csr(rl_engine* e, uint64_t n, const uint32_t* off, const rl_counter* ctrs, const uint64_t* delta,
                     const uint64_t* now, int mem, CsrDev& d) {
    if (!off || !delta || !now) return fail(e, RL_FATAL, "null CSR arrays");
    if (mem == RL_MEM_DEVICE) {
        uint32_t last = 0;
        RL_CUDA(e, cudaMemcpyAsync(&last, off + n, 4, cudaMemcpyDeviceToHost, e->stream));
        RL_CUDA(e, cudaStreamSynchronize(e->stream));
        d.off = off;
        d.ctrs = ctrs;
        d.delta = delta;
        d.now = now;
        d.total = last;
    } else {
        d.total = off[n];
        for (uint64_t i = 0; i < n; i++)
            if (now[i] == 0)
                return fail(e, RL_FATAL, "now_us[%llu] must be >= 1 — the call was refused before the table was touched",
                            (unsigned long long)i);
        if (d.total > e->max_counters)
            return fail(e, RL_FATAL, "batch has %llu counters > max_counters=%u", (unsigned long long)d.total, e->max_counters);
        RL_CUDA(e, e->d_in_off.reserve(e->max_batch + 1));
        RL_CUDA(e, e->d_in_ctrs.reserve(e->max_counters));
        RL_CUDA(e, e->d_in_delta.reserve(e->max_batch));
        RL_CUDA(e, e->d_in_now.reserve(e->max_batch));
        RL_CUDA(e, cudaMemcpyAsync(e->d_in_off.p, off, (n + 1) * 4, cudaMemcpyHostToDevice, e->stream));
        if (d.total)
            RL_CUDA(e, cudaMemcpyAsync(e->d_in_ctrs.p, ctrs, d.total * sizeof(rl_counter), cudaMemcpyHostToDevice, e->stream));
        RL_CUDA(e, cudaMemcpyAsync(e->d_in_delta.p, delta, n * 8, cudaMemcpyHostToDevice, e->stream));
        RL_CUDA(e, cudaMemcpyAsync(e->d_in_now.p, now, n * 8, cudaMemcpyHostToDevice, e->stream));
        d.off = e->d_in_off.p;
        d.ctrs = e->d_in_ctrs.p;
        d.delta = e->d_in_delta.p;
        d.now = e->d_in_now.p;
    }
    if (d.total > e->max_counters)
        return fail(e, RL_FATAL, "batch has %llu counters > max_counters=%u", (unsigned long long)d.total, e->max_counters);
    return RL_OK;
}

int rl_check_and_update_batch(rl_engine* e, uint64_t n, const uint32_t* ctr_off, const rl_counter* ctrs,
                              const uint64_t* delta, const uint64_t* now_us, int load_counters, int mem,
                              uint8_t* out_limited, uint32_t* out_first_limited, uint64_t* out_remaining,
                              uint64_t* out_ttl_us) {
    int r = ensure_ready(e, n);
    if (r) return r;
    if (n == 0) return RL_OK;
    if (!out_limited) return fail(e, RL_FATAL, "null out_limited");
    CsrDev c;
    if ((r = stage_csr(e, n, ctr_off, ctrs, delta, now_us, mem, c))) return r;
    const bool lc = load_counters && (out_remaining || out_ttl_us);
    e->stats.batches++;
    e->stats.requests += n;
    Outs o;
    if (mem == RL_MEM_DEVICE) {
        o.limited = out_limited;
        o.first = out_first_limited;
        o.rem = lc ? out_remaining : nullptr;
        o.ttl = lc ? out_ttl_us : nullptr;
    } else {
        if ((r = stage_outs(e, n, c.total, out_first_limited != nullptr, lc, o))) return r;
    }
    o.off = c.off;
    RlDev D = make_dev(e);
    RlResolveOut O{e->d_acc.p, nullptr, nullptr, o.limited, o.first};
    k_resolve_csr<<<ceil_div(n, 128), 128, 0, e->stream>>>(D, (uint32_t)n, c.off, c.ctrs, c.now, O, 1);
    RL_LAUNCH_CHECK(e);
    if ((r = check_resolve_error(e))) return r;
    if (c.total) {
        if ((r = run_acc_pipeline(e, (uint32_t)c.total, (uint32_t)n, c.delta, c.now, 0, load_counters ? 1 : 0, o))) return r;
    }
    if (mem == RL_MEM_HOST) {
        RL_CUDA(e, cudaMemcpyAsync(out_limited, o.limited, n, cudaMemcpyDeviceToHost, e->stream));
        if (out_first_limited)
            RL_CUDA(e, cudaMemcpyAsync(out_first_limited, o.first, n * 4, cudaMemcpyDeviceToHost, e->stream));
        if (lc && out_remaining && c.total)
            RL_CUDA(e, cudaMemcpyAsync(out_remaining, o.rem, c.total * 8, cudaMemcpyDeviceToHost, e->stream));
        if (lc && out_ttl_us && c.total)
            RL_CUDA(e, cudaMemcpyAsync(out_ttl_us, o.ttl, c.total * 8, cudaMemcpyDeviceToHost, e->stream));
        return check_device_error(e);
    }
    return RL_OK;
}

int rl_update_batch(rl_engine* e, uint64_t n, const uint32_t* ctr_off, const rl_counter* ctrs, const uint64_t* delta,
                    const uint64_t* now_us, int mem) {
    int r = ensure_ready(e, n);
    if (r) return r;
    if (n == 0) return RL_OK;
    CsrDev c;
    if ((r = stage_csr(e, n, ctr_off, ctrs, delta, now_us, mem, c))) return r;
    e->stats.batches++;
    e->stats.requests += n;
    if (c.total == 0) return RL_OK;
    Outs o;
    RlDev D = make_dev(e);
    RlResolveOut O{e->d_acc.p, nullptr, nullptr, nullptr, nullptr};
    k_resolve_csr<<<ceil_div(n, 128), 128, 0, e->stream>>>(D, (uint32_t)n, c.off, c.ctrs, c.now, O, 0);
    RL_LAUNCH_CHECK(e);
    if ((r = check_resolve_error(e))) return r;
    if ((r = run_acc_pipeline(e, (uint32_t)c.total, (uint32_t)n, c.delta, c.now, 2, 0, o))) return r;
    if (mem == RL_MEM_HOST) return check_device_error(e);
    return RL_OK;
}

int rl_update_records(rl_engine* e, uint64_t n, const rl_record* recs, int mem) {
    int r = ensure_ready(e, n, mem != RL_MEM_DEVICE);
    if (r) return r;
    if (n == 0) return RL_OK;
    if (!recs) return fail(e, RL_FATAL, "null recs");
    e->stats.batches++;
    e->stats.requests += n;
    const rl_record* d_recs = recs;
    if (mem == RL_MEM_HOST) {
        RL_CUDA(e, e->d_in_recs.reserve(e->max_batch));
        RL_CUDA(e, cudaMemcpyAsync(e->d_in_recs.p, recs, n * sizeof(rl_record), cudaMemcpyHostToDevice, e->stream));
        d_recs = e->d_in_recs.p;
    }
    Outs o;
    if ((r = run_record_pipeline(e, (uint32_t)n, d_recs, 2, 0, o, mem == RL_MEM_DEVICE))) return r;
    if (mem == RL_MEM_HOST) return check_device_error(e);
    return RL_OK;
}

int rl_is_within_limits_batch(rl_engine* e, uint64_t n, const uint32_t* ctr_off, const rl_counter* ctrs,
                              const uint64_t* delta, const uint64_t* now_us, int mem, uint8_t* out_limited,
                              uint32_t* out_first_limited) {
    int r = ensure_ready(e, n);
    if (r) return r;
    if (n == 0) return RL_OK;
    if (!out_limited) return fail(e, RL_FATAL, "null out_limited");
    CsrDev c;
    if ((r = stage_csr(e, n, ctr_off, ctrs, delta, now_us, mem, c))) return r;
    Outs o;
    if (mem == RL_MEM_DEVICE) {
        o.limited = out_limited;
        o.first = out_first_limited;
    } else if ((r = stage_outs(e, n, 0, out_first_limited != nullptr, false, o))) {
        return r;
    }
    RlDev D = make_dev(e);
    const uint32_t blocks = ceil_div(n, 128);
    switch (e->cells) {
        case 1: k_query_csr<1><<<blocks, 128, 0, e->stream>>>(D, (uint32_t)n, c.off, c.ctrs, c.delta, c.now, o.limited, o.first); break;
        case 3: k_query_csr<3><<<blocks, 128, 0, e->stream>>>(D, (uint32_t)n, c.off, c.ctrs, c.delta, c.now, o.limited, o.first); break;
        default: k_query_csr<7><<<blocks, 128, 0, e->stream>>>(D, (uint32_t)n, c.off, c.ctrs, c.delta, c.now, o.limited, o.first); break;
    }
    RL_LAUNCH_CHECK(e);
    if (mem == RL_MEM_HOST) {
        RL_CUDA(e, cudaMemcpyAsync(out_limited, o.limited, n, cudaMemcpyDeviceToHost, e->stream));
        if (out_first_limited)
            RL_CUDA(e, cudaMemcpyAsync(out_first_limited, o.first, n * 4, cudaMemcpyDeviceToHost, e->stream));
        return check_device_error(e);
    }
    return RL_OK;
}

int rl_is_within_limits_records(rl_engine* e, uint64_t n, const rl_record* recs, int mem, uint8_t* out_limited,
                                uint32_t* out_first_limited) {
    int r = ensure_ready(e, n);
    if (r) return r;
    if (n == 0) return RL_OK;
    if (!recs || !out_limited) return fail(e, RL_FATAL, "null recs/out_limited");
    const rl_record* d_recs = recs;
    Outs o;
    if (mem == RL_MEM_DEVICE) {
        o.limited = out_limited;
        o.first = out_first_limited;
    } else {
        RL_CUDA(e, e->d_in_recs.reserve(e->max_batch));
        RL_CUDA(e, cudaMemcpyAsync(e->d_in_recs.p, recs, n * sizeof(rl_record), cudaMemcpyHostToDevice, e->stream));
        d_recs = e->d_in_recs.p;
        if ((r = stage_outs(e, n, 0, out_first_limited != nullptr, false, o))) return r;
    }
    RlDev D = make_dev(e);
    const uint32_t blocks = ceil_div(n, 128);
    switch (e->cells) {
        case 1: k_query_records<1><<<blocks, 128, 0, e->stream>>>(D, (uint32_t)n, d_recs, o.limited, o.first); break;
        case 3: k_query_records<3><<<blocks, 128, 0, e->stream>>>(D, (uint32_t)n, d_recs, o.limited, o.first); break;
        default: k_query_records<7><<<blocks, 128, 0, e->stream>>>(D, (uint32_t)n, d_recs, o.limited, o.first); break;
    }
    RL_LAUNCH_CHECK(e);
    if (mem == RL_MEM_HOST) {
        RL_CUDA(e, cudaMemcpyAsync(out_limited, o.limited, n, cudaMemcpyDeviceToHost, e->stream));
        if (out_first_limited)
            RL_CUDA(e, cudaMemcpyAsync(out_first_limited, o.first, n * 4, cudaMemcpyDeviceToHost, e->stream));
        return check_device_error(e);
    }
    return RL_OK;
}

// ---------------------------------------------------------------------------------------
int rl_bucket_by_owner(rl_engine* e, uint64_t n, const rl_record* d_recs, uint32_t world, rl_record* d_out_recs,
                       uint32_t* d_out_src, uint64_t* h_counts) {
    if (!e) return RL_FATAL;
    if (world == 0 || world > 32) return fail(e, RL_FATAL, "world must be 1..32");
    RL_CUDA(e, cudaSetDevice(e->device));
    for (uint32_t w = 0; w < world; w++) h_counts[w] = 0;
    if (n == 0) return RL_OK;
    uint32_t tile = ceil_div(n, kMaxTiles);
    tile = std::max<uint32_t>(512, ((tile + 255) / 256) * 256);
    const uint32_t num_tiles = ceil_div(n, tile);
    RL_CUDA(e, e->d_bucket.reserve((size_t)(kMaxTiles + 1) * 32 + 32));
    RL_CUDA(e, e->d_bucket_counts.reserve(32));
    uint32_t* tile_cnt = e->d_bucket.p;
    uint32_t* owner_base = e->d_bucket.p + (size_t)(kMaxTiles + 1) * 32;
    k_bucket<false><<<num_tiles, RL_PART_THREADS, 0, e->stream>>>(d_recs, (uint32_t)n, world, tile, tile_cnt, owner_base,
                                                                  d_out_recs, d_out_src, 0, nullptr);
    RL_LAUNCH_CHECK(e);
    k_bucket_scan<<<1, 32, 0, e->stream>>>(num_tiles, world, tile_cnt, owner_base, e->d_bucket_counts.p, 0, nullptr);
    RL_LAUNCH_CHECK(e);
    k_bucket<true><<<num_tiles, RL_PART_THREADS, 0, e->stream>>>(d_recs, (uint32_t)n, world, tile, tile_cnt, owner_base,
                                                                 d_out_recs, d_out_src, 0, nullptr);
    RL_LAUNCH_CHECK(e);
    unsigned long long counts[32];
    RL_CUDA(e, cudaMemcpyAsync(counts, e->d_bucket_counts.p, world * sizeof(unsigned long long), cudaMemcpyDeviceToHost,
                               e->stream));
    RL_CUDA(e, cudaStreamSynchronize(e->stream));
    for (uint32_t w = 0; w < world; w++) h_counts[w] = counts[w];
    return RL_OK;
}

int rl_bucket_by_owner_padded(rl_engine* e, uint64_t n, const rl_record* d_recs, uint32_t world, uint32_t slot_cap,
                              rl_record* d_out_recs, uint32_t* d_out_pos, uint32_t* d_overflow) {
    if (!e) return RL_FATAL;
    if (world == 0 || world > 32 || slot_cap == 0) return fail(e, RL_FATAL, "world must be 1..32 and slot_cap > 0");
    RL_CUDA(e, cudaSetDevice(e->device));
    if (n == 0) return RL_OK;
    uint32_t tile = ceil_div(n, kMaxTiles);
    tile = std::max<uint32_t>(512, ((tile + 255) / 256) * 256);
    const uint32_t num_tiles = ceil_div(n, tile);
    RL_CUDA(e, e->d_bucket.reserve((size_t)(kMaxTiles + 1) * 32 + 32));
    RL_CUDA(e, e->d_bucket_counts.reserve(32));
    uint32_t* tile_cnt = e->d_bucket.p;
    uint32_t* owner_base = e->d_bucket.p + (size_t)(kMaxTiles + 1) * 32;
    // unused slots = no-op records (ns_id 0xFFFFFFFF: a namespace without limits)
    RL_CUDA(e, cudaMemsetAsync(d_out_recs, 0xFF, (size_t)world * slot_cap * sizeof(rl_record), e->stream));
    k_bucket<false><<<num_tiles, RL_PART_THREADS, 0, e->stream>>>(d_recs, (uint32_t)n, world, tile, tile_cnt, owner_base,
                                                                  d_out_recs, nullptr, slot_cap, d_out_pos);
    RL_LAUNCH_CHECK(e);
    k_bucket_scan<<<1, 32, 0, e->stream>>>(num_tiles, world, tile_cnt, owner_base, e->d_bucket_counts.p, slot_cap,
                                           d_overflow);
    RL_LAUNCH_CHECK(e);
    k_bucket<true><<<num_tiles, RL_PART_THREADS, 0, e->stream>>>(d_recs, (uint32_t)n, world, tile, tile_cnt, owner_base,
                                                                 d_out_recs, nullptr, slot_cap, d_out_pos);
    RL_LAUNCH_CHECK(e);
    return RL_OK;
}

int rl_gather_u8(rl_engine* e, uint64_t n, const uint8_t* d_in, const uint32_t* d_pos, uint8_t* d_out) {
    if (!e) return RL_FATAL;
    RL_CUDA(e, cudaSetDevice(e->device));
    if (n == 0) return RL_OK;
    k_gather_u8<<<ceil_div(n, 256), 256, 0, e->stream>>>((uint32_t)n, d_in, d_pos, d_out);
    RL_LAUNCH_CHECK(e);
    return RL_OK;
}

int rl_record_lane_put(rl_engine* e, uint64_t n_slots, rl_record* d_recs, const uint8_t* d_lane) {
    if (!e) return RL_FATAL;
    RL_CUDA(e, cudaSetDevice(e->device));
    if (n_slots == 0) return RL_OK;
    k_lane_put<<<ceil_div(n_slots, 256), 256, 0, e->stream>>>((uint32_t)n_slots, d_recs, d_lane);
    RL_LAUNCH_CHECK(e);
    return RL_OK;
}

int rl_record_lane_gather(rl_engine* e, uint64_t n, const rl_record* d_recs, const uint32_t* d_pos, uint8_t* d_out) {
    if (!e) return RL_FATAL;
    RL_CUDA(e, cudaSetDevice(e->device));
    if (n == 0) return RL_OK;
    k_lane_gather<<<ceil_div(n, 256), 256, 0, e->stream>>>((uint32_t)n, d_recs, d_pos, d_out);
    RL_LAUNCH_CHECK(e);
    return RL_OK;
}

int rl_unpermute_u8(rl_engine* e, uint64_t n, const uint8_t* d_in, const uint32_t* d_src, uint8_t* d_out) {
    if (!e) return RL_FATAL;
    RL_CUDA(e, cudaSetDevice(e->device));
    if (n == 0) return RL_OK;
    k_unpermute_u8<<<ceil_div(n, 256), 256, 0, e->stream>>>((uint32_t)n, d_in, d_src, d_out);
    RL_LAUNCH_CHECK(e);
    return RL_OK;
}

#include "rl_shard_host.inc"

}  // extern "C"

// ---- what rl_maint.cu may do with an engine (rl_internal.h) -------------------------------------------------------------
int rl_internal_view(rl_engine* e, RlTableView* out) {
    if (!e || !out) return RL_FATAL;
    RL_CUDA(e, cudaSetDevice(e->device));
    int r = pipe_fence(e);
    if (r) return r;
    r = upload_tables(e);
    if (r) return r;
    out->rows = e->d_rows;
    out->cells = e->cells;
    out->log2P = e->log2P;
    out->log2R = e->log2R;
    out->row_bytes = e->row_bytes;
    out->capacity = e->capacity;
    out->ns_cap = e->ns_cap;
    out->limits_cap = e->limits_cap;
    out->stream = e->stream;
    out->device = e->device;
    return RL_OK;
}
int rl_internal_fail(rl_engine* e, int status, const char* msg) { return fail(e, status, "%s", msg); }
void rl_internal_launched(rl_engine* e, uint32_t kernels) {
    if (e) e->stats.kernel_launches += kernels;
}
void** rl_internal_ext(rl_engine* e, void (*ext_free)(void*)) {
    e->ext_free = ext_free;
    return &e->ext;
}
void rl_internal_set_ns_hook(rl_engine* e, rl_ns_hook_fn fn) { e->ns_hook = fn; }
int rl_internal_reset_hot_rows(rl_engine* e) {
    RL_CUDA(e, cudaMemsetAsync(e->d_hot.p, 0xFF, (RL_HOT_SLOTS + RL_HOT_CAND) * sizeof(uint32_t), e->stream));
    RL_CUDA(e, cudaMemsetAsync(e->d_hot.p + RL_HOT_SLOTS + RL_HOT_CAND, 0, 4 * sizeof(uint32_t), e->stream));
    return RL_OK;
}
