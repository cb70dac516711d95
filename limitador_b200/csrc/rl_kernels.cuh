// rl_kernels.cuh — hand-written sm_100a kernels of the batched rate-limit engine.
//
// Pipeline for one batch (DESIGN.md §3), two launches:
//   k_front : every access finds (or claims) its table row — the one random HBM access of the batch —
//             and every tile (CTA) lays its accesses out by table region inside its own slice of the
//             partition arrays, stream order kept; the LAST block to finish builds the work items
//   k_main  : one CTA per work item; merges the tiles' runs of its region, gathers the 32-B records of
//             its chunk, groups the accesses by table row in shared memory and replays every row's
//             requests in stream order (fixed-window check / increment), so the result equals
//             one-at-a-time execution on the reference InMemoryStorage
//             (limitador/src/storage/in_memory.rs:72-156).
// A region (contiguous slab of rows) is touched by exactly one CTA at a time, and a row by exactly
// one group, so counter values need no atomics at all; the only atomic on the table is the
// 128-bit CAS that claims an empty row for a new key.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/rl_engine.h"
#include "rl_core.h"

#define RL_PART_THREADS 256
#define RL_MAX_TILES 1024  // tiles (CTAs of k_front) per batch: a 1 M-request batch gives every warp one 4-deep probe iteration
// Hot rows (DESIGN.md §3.4): a row that draws a large share of a batch gets a partition of its own and is
// replayed by one CTA of k_hot over its whole request list, instead of being chopped into chained chunks.
#define RL_HOT_SLOTS 256   // rows that can be hot at a time (= threads of k_front's last block)
#define RL_HOT_CAND 128    // candidates k_main can report per batch
#define RL_HOT_THREADS 512
#ifndef RL_HOT_MIN
#define RL_HOT_MIN 32      // a row with this many requests in one k_main chunk becomes a candidate
#endif
#ifndef RL_HOT_KEEP
#define RL_HOT_KEEP 24     // a hot row with fewer requests than this in a batch is dropped again
#endif
#define RL_PART_WARPS (RL_PART_THREADS / 32)
#define RL_PROBE_THREADS 1024
#define RL_IDENT_POSORIG 0x0654321006543210ull
#define RL_ROW_NONE 0xFFFFFFFFu   // row_of: the access has no row (namespace without limits)
#define RL_ROW_ERROR 0xFFFFFFFEu  // row_of: the access could not be evaluated (error flagged)

struct RlDev {
    uint8_t* rows;
    uint32_t log2P;  // regions
    uint32_t log2R;  // rows per region
    const RlCellDesc* desc;  // [ngroups][8]
    const RlLimitDev* limits;
    uint32_t limits_cap;
    const RlNsDev* ns;
    uint32_t ns_cap;
    const uint32_t* ns_limit_ids;
    uint32_t* err;    // sticky max of RL_DEV_*
    uint32_t* flags;  // bit0: batch has multi-row requests
    unsigned long long* kstats;   // nullptr = no accounting; [0] chunks, [1] replay rounds, [2] chained chunks, [3] ordered chunks
    uint32_t* hot_rows;           // [RL_HOT_SLOTS] table row index of hot slot h, or 0xFFFFFFFF; rewritten by k_front's tail
    uint32_t* hot_cand;           // [RL_HOT_CAND] rows k_main saw dominate a chunk
    uint32_t* hot_cand_n;
    uint4* trace;                 // nullptr = no tracing (RL_FLAG_TRACE): ring of {event id, call seq, globaltimer lo, hi}
    uint32_t* trace_pos;
    uint32_t seq;                 // call sequence number stamped into the events of this launch
};

// Device-side event trace (RL_FLAG_TRACE, rl_trace_dump): kernels stamp the GPU's nanosecond timer at their
// first block's start and at their last block's end, so that the timeline of a pipelined step — which
// spans several streams and, for sharded steps, several GPUs — can be read without a profiler.
#define RL_TRACE_CAP 65536u
enum { RL_EV_FRONT = 1, RL_EV_MAIN = 2, RL_EV_XCOUNT = 3, RL_EV_XSCATTER = 4, RL_EV_XWAIT = 5, RL_EV_XRETURN = 6,
       RL_EV_XWAITV = 7, RL_EV_XGATHER = 8, RL_EV_HOT = 9 };
__device__ __forceinline__ void rl_trace(uint4* trace, uint32_t* pos, uint32_t ev, uint32_t end, uint32_t seq) {
    if (trace == nullptr) return;
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    const uint32_t i = atomicAdd(pos, 1u) & (RL_TRACE_CAP - 1);
    trace[i] = make_uint4(ev | (end << 8), seq, (uint32_t)t, (uint32_t)(t >> 32));
}

struct RlBatch {
    uint32_t n_acc;          // accesses of this batch (upper bound when n_dev != nullptr)
    uint32_t n_req;
    const uint32_t* n_dev;   // nullable: the access count lives on the device (peer exchange: the inbox fill)
    // partition workspace
    uint32_t* tile_loc;      // [num_tiles][P+2] offset of partition r's run inside tile t's slice of part_idx/part_row
    uint32_t* region_total;  // [P+1] accumulated by the front's tiles; zero between batches
    uint32_t* row_of;        // [n_acc] table row (index) of access a, probed / claimed in pass 1 of k_front
    uint32_t* part_idx;      // [num_tiles * tile] access index; tile t's slice holds its accesses partition by partition
    uint32_t* part_row;      // [num_tiles * tile] its table row
    uint32_t* scan_ctr;      // blocks-done counter of k_front
    uint32_t* ticket;        // work-item ticket of k_main
    uint32_t* exit_ctr;      // CTAs of k_main that found the ticket exhausted (the last one re-arms it)
    uint32_t nhot;           // 0, or RL_HOT_SLOTS: partitions nparts .. nparts+nhot-1 hold one hot row each
    uint32_t nparts;         // partitions of this batch: table regions merged 2^part_shift at a time, so
    uint32_t part_shift;     //   that a small batch still fills its k_main chunks (nparts = P >> part_shift)
    uint32_t tile;           // accesses per tile (multiple of 256)
    uint32_t num_tiles;
    // outputs (device)
    // Sharded steps: the verdict of inbox access `req` goes straight back to its SOURCE rank's verdict inbox
    // (a peer store over NVLink): request index -> (source block, position) through the inbox prefix.
    const uint32_t* omap_prefix;  // nullptr = plain out_limited[req]; else [omap_n + 1] exclusive prefix of the block fills
    uint32_t omap_n;
    uint32_t omap_stride;         // out_limited is then a mirror of the sources' verdict blocks: [omap_n][omap_stride]
    uint8_t* out_limited;
    uint32_t* out_first_limited;
    uint64_t* out_remaining;
    uint64_t* out_ttl;
    const uint32_t* out_off;  // CSR: per-request base index of remaining/ttl; null => req*out_stride
    uint32_t out_stride;
    // coupled (multi-row) requests
    uint32_t* fl_prev;
    uint32_t* fl_next;
    int phase;          // RL_PHASE_*
    int load_counters;  // 0/1
    // work items of k_main (built by the front's last block): x = partition, y/z = [lo, hi) in the partition's list,
    // w = RL_NONE_U32 for a light partition (its chunks run one after the other in one CTA) or the
    // chunk's index inside a heavy partition (one CTA per chunk, committed in order, see k_main)
    uint4* items;
    uint32_t* n_items;
    uint32_t* chain_status;     // [items] 0 none, 1 read set published, 4 committed
    uint32_t* chain_wcnt;       // [items] size of the chunk's published set
    uint32_t* chain_w;          // [items][chunk] rows the chunk touches (bit 0: it writes the row)
    uint32_t heavy_len;         // partitions longer than this are chained; 0xFFFFFFFF disables
    uint32_t chunk;             // accesses per chunk (= k_main block size)
    // undo log of the rows a coupled batch touches (RL_PHASE_SNAPSHOT / k_restore)
    uint8_t** log_row;     // [n_acc] row pointer logged at the partition position of a key's first access
    ulonglong2* log_state; // [n_acc][CELLS]
};

__device__ __forceinline__ void rl_store_verdict(const RlBatch& B, uint32_t req, uint8_t v) {
    if (B.omap_prefix == nullptr) {
        B.out_limited[req] = v;
        return;
    }
    uint32_t s = 0;
    while (s + 1 < B.omap_n && req >= __ldg(B.omap_prefix + s + 1)) s++;
    B.out_limited[(size_t)s * B.omap_stride + (req - __ldg(B.omap_prefix + s))] = v;
}

// k_main phases.  COMMIT: rows and outputs are written (the normal, single pass).
// Coupled batches (requests spanning several rows) run SNAPSHOT once (log the original
// state of every touched row), then SPEC rounds (rows written, outputs not, fl_next
// accumulated; k_restore puts the rows back after each), then COMMIT.
#define RL_PHASE_COMMIT 0
#define RL_PHASE_SPEC 1
#define RL_PHASE_SNAPSHOT 2

// ---------------------------------------------------------------------------------------
// memory helpers: table traffic bypasses L1 (.cg) — rows have no L1 reuse and .cg keeps the
// CTA's own earlier writes (previous chunk) visible without relying on L1 invalidation.
__device__ __forceinline__ ulonglong2 rl_ld_cg(const void* p) {
    return __ldcg(reinterpret_cast<const ulonglong2*>(p));
}
__device__ __forceinline__ void rl_st_cg(void* p, unsigned long long a, unsigned long long b) {
    __stcg(reinterpret_cast<ulonglong2*>(p), make_ulonglong2(a, b));
}
// 128-bit compare-and-swap (PTX atom.cas.b128, sm_90+): claims a row header atomically.
__device__ __forceinline__ ulonglong2 rl_cas128(void* addr, ulonglong2 cmp, ulonglong2 val) {
    ulonglong2 old;
    asm volatile(
        "{\n\t"
        ".reg .b128 c, v, o;\n\t"
        "mov.b128 c, {%3, %4};\n\t"
        "mov.b128 v, {%5, %6};\n\t"
        "atom.global.cas.b128 o, [%2], c, v;\n\t"
        "mov.b128 {%0, %1}, o;\n\t"
        "}\n"
        : "=l"(old.x), "=l"(old.y)
        : "l"(addr), "l"(cmp.x), "l"(cmp.y), "l"(val.x), "l"(val.y)
        : "memory");
    return old;
}
// streaming (read-once) loads of request data: keep them out of L1
__device__ __forceinline__ ulonglong2 rl_ld_stream(const void* p) {
    return __ldcs(reinterpret_cast<const ulonglong2*>(p));
}
__device__ __forceinline__ void rl_set_err(const RlDev& D, uint32_t code) { atomicMax(D.err, code); }

template <int CELLS>
struct RlGeom {
    static constexpr uint32_t ROW_BYTES = 16u * (1 + CELLS);
};

__device__ __forceinline__ uint64_t rl_region_of(const RlDev& D, uint64_t h) {
    return D.log2P ? (h >> (64 - D.log2P)) : 0ull;
}

// Find the row of (key_lo, hdr_hi); optionally claim an empty/tombstoned row for it.
// Linear probing confined to the key's region.  Returns nullptr when absent (and !create)
// or when the region is full (error flagged).
template <int CELLS>
__device__ uint8_t* rl_probe(const RlDev& D, uint64_t h, uint64_t key_lo, uint64_t hdr_hi, bool create) {
    constexpr uint32_t RB = RlGeom<CELLS>::ROW_BYTES;
    const uint32_t R = 1u << D.log2R;
    const uint64_t base = rl_region_of(D, h) << D.log2R;
    const uint32_t idx = (uint32_t)h & (R - 1);
    int tomb = -1;
    uint32_t restarts = 0;
    for (uint32_t i = 0; i < R;) {
        uint8_t* row = D.rows + (base + ((idx + i) & (R - 1))) * RB;
        const ulonglong2 hdr = rl_ld_cg(row);
        if (hdr.x == key_lo && hdr.y == hdr_hi) return row;
        if (hdr.x == 0 && hdr.y == 0) {
            if (!create) return nullptr;
            uint8_t* target = row;
            ulonglong2 expect = make_ulonglong2(0ull, 0ull);
            if (tomb >= 0) {
                target = D.rows + (base + ((idx + (uint32_t)tomb) & (R - 1))) * RB;
                expect = make_ulonglong2(0ull, RL_TOMB_HI);
            }
            const ulonglong2 old = rl_cas128(target, expect, make_ulonglong2(key_lo, hdr_hi));
            if (old.x == expect.x && old.y == expect.y) return target;
            // another prober took the row first: rescan
            if (++restarts > 4 * R) break;
            tomb = -1;
            i = 0;
            continue;
        }
        if (hdr.y == RL_TOMB_HI && tomb < 0) tomb = (int)i;
        i++;
    }
    if (create) {
        if (tomb >= 0) {
            uint8_t* target = D.rows + (base + ((idx + (uint32_t)tomb) & (R - 1))) * RB;
            const ulonglong2 old = rl_cas128(target, make_ulonglong2(0ull, RL_TOMB_HI),
                                             make_ulonglong2(key_lo, hdr_hi));
            if (old.x == 0ull && old.y == RL_TOMB_HI) return target;
        }
        rl_set_err(D, RL_DEV_TABLE_FULL);
    }
    return nullptr;
}

template <int CELLS>
__device__ __forceinline__ void rl_row_load(const uint8_t* row, uint32_t ncells, RlRow<CELLS>& r) {
#pragma unroll
    for (int c = 0; c < CELLS; c++) {
        if ((uint32_t)c < ncells && row) {
            const ulonglong2 v = rl_ld_cg(row + 16 + 16 * c);
            r.value[c] = v.x;
            r.expiry[c] = v.y;
        } else {
            r.value[c] = 0;
            r.expiry[c] = 0;
        }
    }
}
template <int CELLS>
__device__ __forceinline__ void rl_row_store(uint8_t* row, uint32_t dirty, const RlRow<CELLS>& r) {
#pragma unroll
    for (int c = 0; c < CELLS; c++)
        if (dirty & (1u << c)) rl_st_cg(row + 16 + 16 * c, r.value[c], r.expiry[c]);
}

// ---------------------------------------------------------------------------------------
// Access sources.  RecordSrc: access == request, derived on the fly from the 32-B record
// and the namespace table (every namespace is single-row).  AccSrc: materialised accesses
// written by a resolve kernel (general CSR form, or records of multi-row namespaces).
// k_main gathers its chunk straight from the source (one 32-B sector per access): `raw`
// issues the loads, `decode` consumes them — the kernel puts its grouping barrier in between.
struct RlRaw {
    ulonglong2 w0, w1;
};
struct RlReq {       // what the replay needs of an access
    uint32_t req;    // request index (outputs)
    uint32_t cells;  // packed cell list (rl_core.h)
    uint32_t group;  // row group: selects the RlCellDesc block
    uint64_t posorig;
    uint64_t delta, now;
};

// Segmented record source (peer exchange): the owner's inbox holds one fixed-size block per source
// rank, block s filled with seg_prefix[s+1]-seg_prefix[s] records; access a of the batch is the
// (a - seg_prefix[s])-th record of block s.  seg_prefix == nullptr: a plain array.
struct RecordSrc {
    static constexpr bool kAccessIsRequest = true;
    static constexpr bool kCanBeMulti = false;  // every namespace maps to one row
    const rl_record* recs;
    const uint32_t* seg_prefix;  // [nseg+1] exclusive prefix of the block fills (device), or nullptr
    uint32_t nseg;
    uint32_t seg_stride;         // records per block
    // compact != 0: recs points at 16-byte rl_record16 (word0 = ns_id:24 | hits:8 | key_hi:32, word1 = key_lo)
    // and every request carries the batch's one clock reading now_all (a batching front stamps a batch once)
    uint32_t compact;
    uint64_t now_all;
    __device__ __forceinline__ const rl_record* at(uint32_t a) const {
        if (seg_prefix == nullptr) return recs + a;
        uint32_t s = 0;
        while (s + 1 < nseg && a >= __ldg(seg_prefix + s + 1)) s++;
        return recs + (size_t)s * seg_stride + (a - __ldg(seg_prefix + s));
    }
    __device__ __forceinline__ const ulonglong2* at16(uint32_t a) const {
        return reinterpret_cast<const ulonglong2*>(recs) + a;
    }
    // identity of access a: 1 = a row; 0 = no row (namespace without limits: allowed, lib.rs:434-440);
    // -1 = malformed request (error flagged; its verdict byte becomes RL_VERDICT_ERROR, never a silent allow)
    __device__ __forceinline__ int ident(const RlDev& D, uint32_t a, uint64_t& key_lo, uint64_t& hdr_hi) const {
        ulonglong2 w0;
        uint32_t ns_id;
        unsigned long long key_hi = 0;
        const rl_record* r = nullptr;
        if (compact) {
            w0 = rl_ld_stream(at16(a));
            ns_id = (uint32_t)w0.x & 0x00FFFFFFu;
            key_hi = w0.x >> 32;
        } else {
            r = at(a);
            w0 = rl_ld_stream(r);  // ns_id|hits, key_lo
            ns_id = (uint32_t)w0.x;
        }
        if (ns_id >= D.ns_cap) return 0;
        const RlNsDev ns = D.ns[ns_id];
        if (ns.mode != 1) return 0;
        if (!compact) {
            const ulonglong2 w1 = rl_ld_stream(reinterpret_cast<const ulonglong2*>(r) + 1);  // key_hi, now_us
            if (w1.y == 0) {  // 1 <= now_us: a cell stored at expiry 0 would read as absent
                rl_set_err(D, RL_DEV_CLOCK);
                return -1;
            }
            key_hi = w1.x & RL_RECORD_KEY_HI_MASK;
        }
        if (ns.qualified_row) {
            if (!compact && (key_hi >> 32)) {
                rl_set_err(D, RL_DEV_KEY_RANGE);
                return -1;
            }
            key_lo = w0.y;
            hdr_hi = ((uint64_t)ns.group << 32) | key_hi;
        } else {
            key_lo = 0;
            hdr_hi = (uint64_t)ns.group << 32;
        }
        return 1;
    }
    __device__ __forceinline__ RlRaw raw(uint32_t a) const {
        RlRaw w;
        if (compact) {
            w.w0 = rl_ld_stream(at16(a));
            w.w1 = make_ulonglong2(0ull, 0ull);
            return w;
        }
        const rl_record* r = at(a);
        w.w0 = rl_ld_stream(r);
        w.w1 = rl_ld_stream(reinterpret_cast<const ulonglong2*>(r) + 1);
        return w;
    }
    __device__ __forceinline__ void decode(const RlDev& D, uint32_t a, const RlRaw& w, RlReq& q) const {
        const RlNsDev ns = D.ns[compact ? ((uint32_t)w.w0.x & 0x00FFFFFFu) : (uint32_t)w.w0.x];
        q.req = a;
        q.cells = ns.cells;
        q.group = ns.group;
        q.posorig = RL_IDENT_POSORIG;
        q.delta = compact ? ((w.w0.x >> 24) & 0xFFull) : (uint64_t)(w.w0.x >> 32);
        q.now = compact ? now_all : w.w1.y;
    }
};

struct AccSrc {
    static constexpr bool kAccessIsRequest = false;
    static constexpr bool kCanBeMulti = true;
    const RlAccess* acc;
    const uint64_t* delta;  // per request
    const uint64_t* now;    // per request
    __device__ __forceinline__ int ident(const RlDev&, uint32_t a, uint64_t& key_lo, uint64_t& hdr_hi) const {
        const ulonglong2 w0 = rl_ld_stream(&acc[a]);
        key_lo = w0.x;
        hdr_hi = w0.y;
        return hdr_hi != 0 ? 1 : 0;
    }
    __device__ __forceinline__ RlRaw raw(uint32_t a) const {
        RlRaw w;
        w.w0 = rl_ld_stream(&acc[a]);
        w.w1 = rl_ld_stream(reinterpret_cast<const ulonglong2*>(&acc[a]) + 1);
        return w;
    }
    __device__ __forceinline__ void decode(const RlDev&, uint32_t, const RlRaw& w, RlReq& q) const {
        q.req = (uint32_t)w.w1.x;
        q.cells = (uint32_t)(w.w1.x >> 32);
        q.group = (uint32_t)(w.w0.y >> 32);
        q.posorig = w.w1.y;
        q.delta = delta[q.req];
        q.now = now[q.req];
    }
};

// ---------------------------------------------------------------------------------------
// The front kernel: probe + stable partition by table region, one launch.
//
// Tile = a contiguous slice of the batch, one CTA; warp w of the CTA owns the w-th contiguous slice of
// the tile, so stream order == (tile, warp, step, lane).
//   pass 1  every access finds (or, for a new key, claims) its table row — the one random HBM access of
//           the batch, U of them in flight per lane — and the warp counts its accesses per region;
//   layout  the tile's accesses are laid out region by region inside the TILE'S OWN slice of
//           part_idx/part_row (tile_loc[t][r] = offset of region r's run in tile t), so no CTA needs
//           anything from another one: there is no cross-tile prefix and no second kernel.  A region's
//           list is the concatenation over tiles of its runs; k_main merges them on read.
//   pass 2  the same sweep hands out the positions (stable: earlier warps, then rank inside the warp);
//   tail    region totals are accumulated by atomics; the LAST block to finish turns them into the work
//           items of k_main (one global round trip, the rest out of shared memory).
template <int NT>
__device__ __forceinline__ uint32_t rl_block_excl_scan(uint32_t v, uint32_t* s_warp, uint32_t& total) {
    // exclusive prefix of v over the NT threads of the block; s_warp: NT/32 words of shared memory
    constexpr int NW = NT / 32;
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t y = __shfl_up_sync(0xffffffffu, x, o);
        if ((int)lane >= o) x += y;
    }
    if (lane == 31) s_warp[warp] = x;
    __syncthreads();
    uint32_t woff = 0, tot = 0;
#pragma unroll
    for (int w = 0; w < NW; w++) {
        const uint32_t c = s_warp[w];
        if ((uint32_t)w < warp) woff += c;
        tot += c;
    }
    total = tot;
    __syncthreads();  // s_warp may be reused by the caller
    return woff + x - v;
}

__device__ __forceinline__ unsigned long long rl_globaltimer_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

// Tile size: fixed by the host for a host-side count; derived from the device-side count (sharded steps:
// the inbox fill) so that every launched CTA gets its share whatever the fill is.
__device__ __forceinline__ uint32_t rl_tile_of(const RlBatch& B, uint32_t n) {
    if (B.n_dev == nullptr) return B.tile;
    const uint32_t t = (n + B.num_tiles - 1) / B.num_tiles;
    return max(256u, ((t + 255u) / 256u) * 256u);
}
__device__ __forceinline__ uint32_t rl_batch_n(const RlBatch& B) {
    return B.n_dev ? min(*B.n_dev, B.n_acc) : B.n_acc;
}

template <int CELLS, class Src>
__global__ void __launch_bounds__(RL_PART_THREADS) k_front(RlDev D, RlBatch B, Src src) {
    extern __shared__ uint32_t wcnt[];  // [RL_PART_WARPS][P+1] per-warp counts -> positions, then loc[P+2]
    __shared__ uint32_t s_warp[RL_PART_WARPS], s_warp2[RL_PART_WARPS];
    __shared__ uint32_t s_last;
    constexpr uint32_t RB = RlGeom<CELLS>::ROW_BYTES;
    constexpr int U = 4;
    constexpr uint32_t NT = RL_PART_THREADS;
    static_assert(RL_HOT_SLOTS == RL_PART_THREADS, "the tail handles one hot slot per thread");
    __shared__ uint32_t hs_key[2 * RL_HOT_SLOTS], hs_val[2 * RL_HOT_SLOTS];  // row -> hot slot
    const uint32_t nhot = B.nhot;
    const uint32_t P1 = B.nparts + nhot + 1;
    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t tile = blockIdx.x;
    const uint32_t n = rl_batch_n(B);
    const uint32_t tsz = rl_tile_of(B, n);
    const uint32_t t0 = min(tile * tsz, n);
    const uint32_t t1 = min(t0 + tsz, n);
    const uint32_t slice = tsz / RL_PART_WARPS;
    const uint32_t s0 = min(t0 + warp * slice, t1);
    const uint32_t s1 = min(s0 + slice, t1);
    uint32_t* mycnt = wcnt + warp * P1;
    uint32_t* loc = wcnt + RL_PART_WARPS * P1;  // [P1 + 1]
    const uint32_t R = 1u << D.log2R;

    for (uint32_t i = tid; i < RL_PART_WARPS * P1 + P1 + 1; i += NT) wcnt[i] = 0;
    if (tile == 0 && tid == 0) rl_trace(D.trace, D.trace_pos, RL_EV_FRONT, 0, D.seq);
    if (nhot) {
        // the hot-row table of this batch (fixed while the batch is partitioned: every access of a row takes
        // the same route whichever CTA sees it).  A row listed twice resolves to its LOWEST slot everywhere.
        for (uint32_t i = tid; i < 2 * RL_HOT_SLOTS; i += NT) {
            hs_key[i] = 0xFFFFFFFFu;
            hs_val[i] = 0xFFFFFFFFu;
        }
        __syncthreads();
        const uint32_t hr = __ldcg(D.hot_rows + tid);
        if (hr != 0xFFFFFFFFu) {
            uint32_t s2 = (hr * 2654435761u) >> 23;  // 9 bits
            for (;;) {
                const uint32_t old = atomicCAS(&hs_key[s2], 0xFFFFFFFFu, hr);
                if (old == 0xFFFFFFFFu || old == hr) {
                    atomicMin(&hs_val[s2], tid);
                    break;
                }
                s2 = (s2 + 1) & (2 * RL_HOT_SLOTS - 1);
            }
        }
    }
    __syncthreads();
    auto hot_of = [&](uint32_t rowidx) -> uint32_t {
        if (!nhot) return 0xFFFFFFFFu;
        uint32_t s2 = (rowidx * 2654435761u) >> 23;
        for (;;) {
            const uint32_t k = hs_key[s2];
            if (k == rowidx) return hs_val[s2];
            if (k == 0xFFFFFFFFu) return 0xFFFFFFFFu;
            s2 = (s2 + 1) & (2 * RL_HOT_SLOTS - 1);
        }
    };
    auto part_of = [&](uint32_t rowidx) -> uint32_t {
        const uint32_t h = hot_of(rowidx);
        return h != 0xFFFFFFFFu ? B.nparts + h : (rowidx >> D.log2R) >> B.part_shift;
    };

    // ---- pass 1: probe, count ---------------------------------------------------------------------
    for (uint32_t b = s0; b < s1; b += 32 * U) {
        uint64_t klo[U], hhi[U], h[U];
        bool ok[U], bad[U];
        uint8_t* home[U];
        ulonglong2 hdr[U];
#pragma unroll
        for (int u = 0; u < U; u++) {
            const uint32_t a = b + u * 32 + lane;
            klo[u] = hhi[u] = 0;
            const int id = (a < s1) ? src.ident(D, a, klo[u], hhi[u]) : 0;
            ok[u] = id > 0;
            bad[u] = id < 0;
        }
#pragma unroll
        for (int u = 0; u < U; u++) {
            h[u] = rl_row_hash(klo[u], hhi[u]);
            home[u] = D.rows + ((rl_region_of(D, h[u]) << D.log2R) + ((uint32_t)h[u] & (R - 1))) * RB;
            if (ok[u]) hdr[u] = rl_ld_cg(home[u]);  // the home rows of U accesses are fetched together
        }
#pragma unroll
        for (int u = 0; u < U; u++) {
            const uint32_t a = b + u * 32 + lane;
            const bool valid = a < s1;
            uint32_t r = P1 - 1, rowidx = bad[u] ? RL_ROW_ERROR : RL_ROW_NONE;
            if (ok[u]) {
                const uint8_t* row = (hdr[u].x == klo[u] && hdr[u].y == hhi[u])
                                         ? home[u]
                                         : rl_probe<CELLS>(D, h[u], klo[u], hhi[u], true);  // collision chain / insert
                if (row) {
                    rowidx = (uint32_t)((size_t)(row - D.rows) / RB);
                    r = part_of(rowidx);
                } else {
                    rowidx = RL_ROW_ERROR;  // the region is full (error flagged): not evaluated
                }
            }
            if (valid) B.row_of[a] = rowidx;
            const unsigned vmask = __ballot_sync(0xffffffffu, valid);
            if (valid) {
                const unsigned m = __match_any_sync(vmask, r);
                if (lane == (uint32_t)(__ffs(m) - 1)) mycnt[r] += __popc(m);
            }
            __syncwarp();
        }
    }
    __syncthreads();

    // ---- tile-local layout: region r's run starts at loc[r] inside this tile's slice ---------------
    for (uint32_t r = tid; r < P1; r += NT) {
        uint32_t c = 0;
#pragma unroll
        for (int w = 0; w < RL_PART_WARPS; w++) c += wcnt[w * P1 + r];
        loc[r] = c;
    }
    __syncthreads();
    {
        uint32_t carry = 0;
        for (uint32_t base = 0; base < P1; base += NT) {
            const uint32_t i = base + tid;
            const uint32_t v = (i < P1) ? loc[i] : 0;
            uint32_t total;
            const uint32_t ex = rl_block_excl_scan<NT>(v, s_warp, total);
            if (i < P1) {
                loc[i] = carry + ex;
                if (v && i != P1 - 1) atomicAdd(&B.region_total[i], v);
            }
            carry += total;
        }
        if (tid == 0) loc[P1] = carry;
    }
    __syncthreads();
    for (uint32_t r = tid; r < P1; r += NT) {
        uint32_t run = loc[r];
#pragma unroll
        for (int w = 0; w < RL_PART_WARPS; w++) {
            const uint32_t c = wcnt[w * P1 + r];
            wcnt[w * P1 + r] = run;
            run += c;
        }
    }
    for (uint32_t r = tid; r < P1 + 1; r += NT) B.tile_loc[(size_t)tile * (P1 + 1) + r] = loc[r];
    __syncthreads();

    // ---- pass 2: same sweep, now handing out positions ----------------------------------------------
    const size_t tbuf = (size_t)tile * tsz;
    for (uint32_t b = s0; b < s1; b += 32) {
        const uint32_t a = b + lane;
        const bool valid = a < s1;
        uint32_t r = P1 - 1, rowidx = 0xFFFFFFFFu;
        if (valid) {
            rowidx = __ldcg(B.row_of + a);
            if (rowidx < RL_ROW_ERROR) r = part_of(rowidx);
        }
        const unsigned vmask = __ballot_sync(0xffffffffu, valid);
        if (valid) {
            const unsigned m = __match_any_sync(vmask, r);
            const int leader = __ffs(m) - 1;
            uint32_t basepos = 0;
            if ((int)lane == leader) {
                basepos = mycnt[r];
                mycnt[r] = basepos + __popc(m);
            }
            basepos = __shfl_sync(m, basepos, leader);
            const uint32_t mypos = basepos + __popc(m & ((1u << lane) - 1));
            if (r != P1 - 1) {
                B.part_idx[tbuf + mypos] = a;
                B.part_row[tbuf + mypos] = rowidx;
            } else if (Src::kAccessIsRequest && B.out_limited) {
                // request without any applicable limit: not limited (lib.rs:434-440); a request that could
                // not be evaluated (malformed key, full table region) says so instead of reading as allowed
                rl_store_verdict(B, a, (rowidx == RL_ROW_ERROR) ? (uint8_t)RL_VERDICT_ERROR : (uint8_t)0);
                if (B.out_first_limited) B.out_first_limited[a] = RL_NONE_U32;
            }
        }
        __syncwarp();
    }

    // ---- last block: work items ---------------------------------------------------------------------
    __threadfence();
    __syncthreads();
    if (tid == 0) s_last = (atomicAdd(B.scan_ctr, 1u) == gridDim.x - 1);
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    const unsigned long long tk0 = (D.kstats != nullptr && tid == 0) ? rl_globaltimer_ns() : 0ull;
    // region lengths into shared memory (re-armed = zeroed for the next batch on the way); loc[] is free now
    const uint32_t P = B.nparts;  // cold partitions: work items of k_main (hot ones belong to k_hot)
    uint32_t hsum = 0, lsum = 0;
    for (uint32_t q = tid; q < P; q += NT) {
        const uint32_t len = __ldcg(&B.region_total[q]);
        B.region_total[q] = 0;
        loc[q] = len;
        if (len > B.heavy_len) hsum += (len + B.chunk - 1) / B.chunk;
        else if (len) lsum += 1;
    }
    uint32_t th, tl;
    uint32_t hb = rl_block_excl_scan<NT>(hsum, s_warp, th);
    uint32_t lb = rl_block_excl_scan<NT>(lsum, s_warp2, tl);
    // chunks of heavy partitions first: they chain in ticket order
    for (uint32_t q = tid; q < P; q += NT) {
        const uint32_t len = loc[q];
        if (len > B.heavy_len) {
            const uint32_t nc = (len + B.chunk - 1) / B.chunk;
            for (uint32_t k = 0; k < nc; k++) {
                B.chain_status[hb] = 0;
                B.items[hb++] = make_uint4(q, k * B.chunk, min((k + 1) * B.chunk, len), k);
            }
        } else if (len) {
            B.items[th + lb++] = make_uint4(q, 0, len, RL_NONE_U32);
        }
    }
    if (nhot) {
        // ---- the hot-row table of the NEXT batch: drop the rows that cooled down, admit the candidates ----
        __shared__ uint32_t s_free[RL_HOT_SLOTS], s_ck[2 * RL_HOT_CAND], s_keep[RL_HOT_SLOTS], s_used;
        const uint32_t h = tid;
        const uint32_t hrow = __ldcg(D.hot_rows + h);
        const uint32_t hlen = __ldcg(&B.region_total[B.nparts + h]);
        B.region_total[B.nparts + h] = 0;
        const bool keep = (hrow != 0xFFFFFFFFu) && hlen >= RL_HOT_KEEP;
        if (!keep && hrow != 0xFFFFFFFFu) D.hot_rows[h] = 0xFFFFFFFFu;
        s_keep[h] = keep ? 1u : 0u;
        for (uint32_t i = tid; i < 2 * RL_HOT_CAND; i += NT) s_ck[i] = 0xFFFFFFFFu;
        if (tid == 0) s_used = 0;
        uint32_t nfree;
        const uint32_t fpos = rl_block_excl_scan<NT>(keep ? 0u : 1u, s_warp, nfree);  // barriers inside
        if (!keep) s_free[fpos] = h;
        __syncthreads();
        const uint32_t ncand = min(__ldcg(D.hot_cand_n), (uint32_t)RL_HOT_CAND);
        if (tid < ncand) {
            const uint32_t c = __ldcg(D.hot_cand + tid);
            const uint32_t hh = (c != 0xFFFFFFFFu) ? hot_of(c) : 0u;
            const bool already = (c == 0xFFFFFFFFu) || (hh != 0xFFFFFFFFu && s_keep[hh]);
            if (!already) {
                uint32_t s2 = (c * 2654435761u) >> 24;  // 8 bits
                bool first = false;
                for (;;) {  // reported by several chunks: one of them admits it
                    const uint32_t old = atomicCAS(&s_ck[s2], 0xFFFFFFFFu, c);
                    if (old == 0xFFFFFFFFu) {
                        first = true;
                        break;
                    }
                    if (old == c) break;
                    s2 = (s2 + 1) & (2 * RL_HOT_CAND - 1);
                }
                if (first) {
                    const uint32_t k = atomicAdd(&s_used, 1u);
                    if (k < nfree) D.hot_rows[s_free[k]] = c;
                }
            }
        }
        __syncthreads();
        if (tid == 0) *D.hot_cand_n = 0;
    }
    if (tid == 0) {
        *B.n_items = th + tl;
        *B.ticket = 0;
        *B.scan_ctr = 0;  // re-arm for the next batch
        if (D.kstats != nullptr) atomicAdd(D.kstats + 16, rl_globaltimer_ns() - tk0);  // ns spent in this tail
        rl_trace(D.trace, D.trace_pos, RL_EV_FRONT, 1, D.seq);
    }
}

// ---------------------------------------------------------------------------------------
// The main kernel.  MODE 0 = check_and_update, MODE 2 = update_counters.
//
// CTAs take work items from an atomic ticket (so every item a CTA may have to wait for is already
// running: the chained commit below is live whatever order the hardware dispatches CTAs in).  A
// partition's accesses (already in stream order) are taken in chunks of CH (one access per thread).
// Per chunk:
//   1. every thread fetches its (access index, table row) pair — prefetched one chunk ahead — and
//      issues the gather of its 32-B record; while that is in flight the CTA groups the accesses by
//      TABLE ROW with a shared-memory hash table (the probe already resolved key -> row, so the
//      32-bit row index is the exact identity of the key: one CAS, no key comparison), and the
//      claimer ("rep") of a row issues the load of the row state;
//   2. every access gets its stable ordinal inside its row group from one packed shared-memory
//      counter per row (8 bits per warp, added warp-aggregated): ordinal order == thread order ==
//      stream order;
//   3. the rep stages the row state in shared memory;
//   4. the group is replayed by ALL its threads in lock-step run-length rounds (rl_core.h,
//      hypotheses A and B; B in closed form for runs of equal deltas) — two barriers per
//      round, one round for a saturated or an unconstrained hot key;
//   5. the rep writes the dirty cells back.
// Counter values never need atomics: a region belongs to one CTA at a time, a row to one group.
template <int CELLS, int CH>
struct RlMainSmem {
    static constexpr int GT = 2 * CH;
    static constexpr int NW = CH / 32;
    static constexpr int PW = (NW + 7) / 8;
    unsigned long long g_packed[GT * PW];  // per row: member count of every warp, 8 bits each
    unsigned long long d_arr[CH];
    unsigned long long s_val[CH * CELLS];  // row state of the group whose rep is thread `gid`
    unsigned long long s_exp[CH * CELLS];
    uint32_t g_row[GT];        // grouping table: row index claimed by CAS; also the chunk's read set
    uint32_t g_rep[GT];
    uint32_t cells_arr[CH];
    uint32_t g_min[2][2][CH];  // [round parity][A|B][gid]
    uint32_t g_flags[CH];      // by gid: bit2 = replay again (chained chunk, state changed under it)
    uint32_t g_dirty[CH];
    uint32_t rflag[GT];        // chained chunks: row of g_row[] is "ordered" (see below)
    uint32_t need_bits[64];    // earlier chunks (bit per chunk) whose commit I must wait for
    uint32_t scan_off[CH];     // dependency scan: offsets of the earlier chunks' sets, CH chunks at a time
    uint32_t scan_w[NW];
    uint32_t w_cnt;
    uint32_t item;
    // followed in dynamic shared memory by t_pfx[num_tiles + 1] (my partition's list: exclusive prefix of its per-tile
    // run lengths) and t_loc[num_tiles] (where each tile's run starts in part_idx/part_row): sized by the batch's
    // tile count, not by RL_MAX_TILES — shared memory a 128-tile batch does not need would come out of k_main's L1
};
template <int CELLS, int CH>
__host__ __device__ constexpr size_t rl_main_smem_bytes(uint32_t num_tiles) {
    return sizeof(RlMainSmem<CELLS, CH>) + (2 * (size_t)num_tiles + 1) * sizeof(uint32_t);
}

// Per-thread view of the limits its access touches, in the access's own cell order.
struct RlMyLimits {
    uint64_t mx[RL_MAX_CELLS];
    uint32_t qmask;  // bit k: k-th touched cell belongs to a qualified limit
};

// Hypotheses A and B for one access against the staged row state (shared memory).
//   a_ok : denied under S and nothing is created / reset / incremented; fl = position of the
//          first limited counter (in_memory.rs:110-112,130-132,141-143)
//   b_ok : every touched cell is live at `now` and stays within its limit after adding
//          `dsum` (this request's delta plus those of the run before it)
template <int CELLS>
__device__ __forceinline__ void rl_eval_ab(const unsigned long long* sv, const unsigned long long* se,
                                           const RlMyLimits& L, uint32_t cells, uint64_t posorig, uint64_t delta,
                                           uint64_t dsum, uint64_t now, bool lc, bool check_limit, bool& a_ok,
                                           bool& b_ok, uint32_t& fl) {
    const uint32_t n = rl_cells_n(cells);
    bool absent_reached = false, live_all = true, within_all = true;
    fl = RL_NONE_U32;
#pragma unroll
    for (int k = 0; k < CELLS; k++) {
        if ((uint32_t)k < n) {
            const uint32_t c = rl_cells_at(cells, k);
            const uint64_t v = sv[c], e = se[c];
            const bool reached = lc || fl == RL_NONE_U32;  // !lc: the walk returns at the first limited counter
            if (reached && ((L.qmask >> k) & 1u) && e == 0) absent_reached = true;
            const uint64_t vv = (e <= now) ? 0 : v;
            if (reached && fl == RL_NONE_U32 && vv + delta > L.mx[k]) fl = rl_pos_at(posorig, k);
            if (e <= now) live_all = false;
            if (v + dsum > L.mx[k]) within_all = false;
        }
    }
    a_ok = (fl != RL_NONE_U32) && !absent_reached;
    b_ok = live_all && (within_all || !check_limit);
}

// With RL_FLAG_KERNEL_STATS (D.kstats != nullptr) k_main accounts its chunks, rounds and SM cycles per
// phase (thread 0, one clock64 and one atomic per phase and chunk): rl_stats.phase_cycles.  It costs a
// few % of a 65536-request step, hence opt-in.
#ifndef RL_MID_CTAS
#define RL_MID_CTAS 5  // resident 128-thread k_main CTAs per SM asked of the compiler for 3..4-cell rows (registers = 512 / this)
#endif
#ifndef RL_WAIT_NS
#define RL_WAIT_NS 100  // back-off of the chained-commit wait loops
#endif
#ifndef RL_KSTATS
#define RL_KSTATS 1  // build with -DRL_KSTATS=0 to compile the accounting out (A/B of its cost)
#endif
#if RL_KSTATS
#define RL_PHASE_TICK(i)                                                         \
    if (D.kstats != nullptr && tid == 0) {                                       \
        const long long tnow = clock64();                                        \
        atomicAdd(D.kstats + 8 + (i), (unsigned long long)(tnow - tph));         \
        tph = tnow;                                                              \
    }
#define RL_KSTAT_ADD(i, v) \
    if (D.kstats != nullptr) atomicAdd(D.kstats + (i), (unsigned long long)(v))
#else
#define RL_PHASE_TICK(i)
#define RL_KSTAT_ADD(i, v)
#endif

// The sequential rule applied by ONE thread directly on the staged row state (shared
// memory) — the default path (single-row request, load_counters off).  Same arithmetic as
// rl_walk_check_single / rl_walk_update (rl_core.h), without a private copy of the row.
//   in_memory.rs:122-127 (insert on lookup), :110-112,130-132 (early return), :146-153 (update)
template <int CELLS>
__device__ __forceinline__ uint32_t rl_apply_check_smem(unsigned long long* sv, unsigned long long* se,
                                                        const RlMyLimits& L, const RlCellDesc* gdesc, uint32_t cells,
                                                        uint64_t posorig, uint64_t delta, uint64_t now,
                                                        uint32_t& dirty) {
    const uint32_t n = rl_cells_n(cells);
    uint32_t fl = RL_NONE_U32;
#pragma unroll
    for (int k = 0; k < CELLS; k++) {
        if ((uint32_t)k < n && fl == RL_NONE_U32) {
            const uint32_t c = rl_cells_at(cells, k);
            uint64_t v = sv[c], e = se[c];
            if (((L.qmask >> k) & 1u) && e == 0) {
                e = now + gdesc[c].window_us;
                v = 0;
                sv[c] = 0;
                se[c] = e;
                dirty |= 1u << c;
            }
            const uint64_t vv = (e <= now) ? 0 : v;
            if (vv + delta > L.mx[k]) fl = rl_pos_at(posorig, k);
        }
    }
    if (fl != RL_NONE_U32) return fl;
#pragma unroll
    for (int k = 0; k < CELLS; k++) {
        if ((uint32_t)k < n) {
            const uint32_t c = rl_cells_at(cells, k);
            if (se[c] <= now) {
                se[c] = now + gdesc[c].window_us;
                sv[c] = delta;
            } else {
                sv[c] += delta;
            }
            dirty |= 1u << c;
        }
    }
    return RL_NONE_U32;
}

template <int CELLS>
__device__ __forceinline__ void rl_apply_update_smem(unsigned long long* sv, unsigned long long* se,
                                                     const RlCellDesc* gdesc, uint32_t cells, uint64_t delta,
                                                     uint64_t now, uint32_t& dirty) {
    const uint32_t n = rl_cells_n(cells);
#pragma unroll
    for (int k = 0; k < CELLS; k++) {
        if ((uint32_t)k < n) {
            const uint32_t c = rl_cells_at(cells, k);
            if (se[c] <= now) {
                se[c] = now + gdesc[c].window_us;
                sv[c] = delta;
            } else {
                sv[c] += delta;
            }
            dirty |= 1u << c;
        }
    }
}

// The lock-step run-length replay of ONE row group by all its member threads (DESIGN.md §3.3), shared by k_main
// (many groups per chunk) and k_hot (one hot row per CTA).  Every thread of the CTA calls it — the rounds
// are separated by CTA barriers — with the view of ITS group:
//   gsv/gse  staged row state of the group (CELLS values / expiries, shared memory)
//   gmin     the group's minima words: gmin[(parity * 2 + {0 A, 1 B}) * gstride], armed to 0xFFFFFFFF
//   gdirty   the group's dirty-cell mask
//   ord/cnt  my stream-order ordinal inside the group and the group's size
//   peers    the lanes of my warp that belong to my group (leader = lowest of them; solo = I am alone)
// Returns the number of rounds the CTA ran.
template <int CELLS, int MODE, bool LC>
__device__ __forceinline__ uint32_t rl_replay_rounds(const RlBatch& B, bool write_out, unsigned long long* gsv,
                                                     unsigned long long* gse, uint32_t* gmin, uint32_t gstride,
                                                     uint32_t* gdirty, const RlReq& acc, const RlMyLimits& L,
                                                     const RlCellDesc* desc, const RlCellDesc* gdesc, bool multi,
                                                     bool like_rep, bool valid, unsigned peers, bool solo, int leader,
                                                     uint32_t lane, uint32_t ord, uint32_t cnt, bool& done, uint32_t& pos) {
    constexpr bool lc = LC;
    const uint64_t delta = acc.delta, now = acc.now;
    const uint32_t ncell = rl_cells_n(acc.cells);
    uint32_t nrounds = 0;
    for (uint32_t round = 0;; round++) {
        nrounds++;
        const uint32_t par = round & 1;
        uint32_t fl = RL_NONE_U32;
        RlRow<CELLS> loc;
        uint32_t amin = 0xFFFFFFFFu, bmin = 0xFFFFFFFFu;  // my ordinal if hypothesis A / B fails for me
        if (!done) {
            bool aok = false, bok = false;
            if (!multi) {
                const uint64_t dsum = (uint64_t)(ord - pos + 1) * delta;
                // update_counters never tests the limit: a run only needs live cells
                rl_eval_ab<CELLS>(gsv, gse, L, acc.cells, acc.posorig, delta, dsum, now, lc, MODE == 0, aok, bok, fl);
                if (MODE == 2) aok = false;
                bok = bok && like_rep;
            }
            if (lc) {
                // remaining/ttl need the state this request sees: copy it before the barrier,
                // the run's last member republishes S right after it
#pragma unroll
                for (int c = 0; c < CELLS; c++) {
                    loc.value[c] = gsv[c];
                    loc.expiry[c] = gse[c];
                }
            }
            if (!aok) amin = ord;
            if (!bok) bmin = ord;
        }
        if (valid) {
            // one shared-memory atomic per (warp, row) instead of one per access
            if (!solo) {
                amin = __reduce_min_sync(peers, amin);
                bmin = __reduce_min_sync(peers, bmin);
            }
            if ((int)lane == leader) {
                if (amin != 0xFFFFFFFFu) atomicMin(&gmin[(par * 2 + 0) * gstride], amin);
                if (bmin != 0xFFFFFFFFu) atomicMin(&gmin[(par * 2 + 1) * gstride], bmin);
            }
        }
        __syncthreads();
        if (!done) {
            const uint32_t mA = min(gmin[(par * 2 + 0) * gstride], cnt);
            const uint32_t mB = min(gmin[(par * 2 + 1) * gstride], cnt);
            uint32_t newpos;
            bool mine = false, store = false, fast_store = false;
            uint32_t dirty = 0;
            uint64_t* rem = nullptr;
            uint64_t* ttl = nullptr;
            if (MODE == 0 && lc && write_out) {
                const size_t ob = B.out_off ? (size_t)B.out_off[acc.req] : (size_t)acc.req * B.out_stride;
                if (B.out_remaining) rem = B.out_remaining + ob;
                if (B.out_ttl) ttl = B.out_ttl + ob;
            }
            if (mA > pos) {  // run of denied requests: state untouched, fl from the evaluation
                newpos = mA;
                if (ord < mA) {
                    mine = true;
                    if (lc && write_out) {  // remaining / ttl of every counter
                        fl = rl_walk_check_single<CELLS>(loc, dirty, desc, acc.cells, acc.posorig, delta, now, true, rem, ttl);
                        dirty = 0;
                    }
                }
            } else if (mB > pos) {  // run of allowed requests with equal deltas: values accumulate
                newpos = mB;
                if (ord < mB) {
                    mine = true;
                    fl = RL_NONE_U32;
                    store = (ord == mB - 1);
                    if (MODE == 0 && lc && write_out) {
                        rl_advance_run<CELLS>(loc, acc.cells, (uint64_t)(ord - pos) * delta);
                        fl = rl_walk_check_single<CELLS>(loc, dirty, desc, acc.cells, acc.posorig, delta, now, lc, rem, ttl);
                        fast_store = false;
                    } else if (store) {
                        // the run's last member is the sole writer of S (nobody reads it until
                        // the next barrier): add the run's deltas in place
                        const uint64_t add = (uint64_t)(mB - pos) * delta;
#pragma unroll
                        for (int k = 0; k < CELLS; k++)
                            if ((uint32_t)k < ncell) {
                                const uint32_t c = rl_cells_at(acc.cells, k);
                                gsv[c] += add;
                                dirty |= 1u << c;
                            }
                        fast_store = true;
                    }
                }
            } else {  // the request at `pos` is applied alone, sequential rule
                newpos = pos + 1;
                if (ord == pos) {
                    mine = true;
                    store = true;
                    if (!lc && !multi) {
                        fast_store = true;  // operate on the staged state in place
                        if (MODE == 2)
                            rl_apply_update_smem<CELLS>(gsv, gse, gdesc, acc.cells,
                                                        delta, now, dirty);
                        else
                            fl = rl_apply_check_smem<CELLS>(gsv, gse, L, gdesc,
                                                            acc.cells, acc.posorig, delta, now, dirty);
                    } else {
                        if (!lc) {
#pragma unroll
                            for (int c = 0; c < CELLS; c++) {
                                loc.value[c] = gsv[c];
                                loc.expiry[c] = gse[c];
                            }
                        }
                        if (MODE == 2) {
                            rl_walk_update<CELLS>(loc, dirty, desc, acc.cells, delta, now);
                        } else if (!multi) {
                            fl = rl_walk_check_single<CELLS>(loc, dirty, desc, acc.cells, acc.posorig, delta, now, lc, rem, ttl);
                        } else {
                            const uint32_t fl_in = B.fl_prev[acc.req];
                            const uint32_t local = rl_walk_check_multi<CELLS>(loc, dirty, desc, acc.cells, acc.posorig,
                                                                             delta, now, lc, fl_in, rem, ttl);
                            if (!write_out && local != RL_NONE_U32) atomicMin(&B.fl_next[acc.req], local);
                            fl = fl_in;
                        }
                    }
                }
            }
            if (mine) {
                done = true;
                if (MODE == 0 && write_out) {
                    rl_store_verdict(B, acc.req, (uint8_t)(fl != RL_NONE_U32));
                    if (B.out_first_limited) {
                        if (fl == RL_NONE_U32) {
                            B.out_first_limited[acc.req] = RL_NONE_U32;
                        } else {
                            // the access holding position fl names the limit
#pragma unroll
                            for (int k = 0; k < CELLS; k++)
                                if ((uint32_t)k < ncell && rl_pos_at(acc.posorig, k) == fl)
                                    B.out_first_limited[acc.req] = desc[rl_cells_at(acc.cells, k)].limit_id;
                        }
                    }
                }
            }
            // the barrier between evaluation and this point ordered every read of S
            // before the publication of the new state
            if (store && dirty) {
                if (!fast_store) {
#pragma unroll
                    for (int c = 0; c < CELLS; c++)
                        if (dirty & (1u << c)) {
                            gsv[c] = loc.value[c];
                            gse[c] = loc.expiry[c];
                        }
                }
                atomicOr(&*gdirty, dirty);
            }
            if (mine && ord == newpos - 1) {  // last finalised member re-arms the group
                gmin[((par ^ 1) * 2 + 0) * gstride] = 0xFFFFFFFFu;
                gmin[((par ^ 1) * 2 + 1) * gstride] = 0xFFFFFFFFu;
            }
            pos = newpos;
        }
        if (!__syncthreads_or(!done)) break;
    }
    return nrounds;
}

template <int GT>
__device__ __forceinline__ uint32_t rl_group_slot(uint32_t row, uint32_t weak) {
    // weak (test aid, RL_FLAG_DEBUG_WEAK_TAGS): four home slots for the whole chunk, so the linear
    // probing of the grouping table is exercised to its full length
    return weak ? (row & 3u) : ((row * 2654435761u) >> 7) & (GT - 1);
}

// GEO = cells per row of the table layout (row bytes), CELLS = cells any row group actually
// uses (<= GEO): loops, registers and shared memory are sized by the latter.
template <int GEO, int CELLS, class Src, int MODE, int CH, bool LC>
__global__ void __launch_bounds__(CH, (CELLS <= 2 ? 8 : (CELLS <= 4 ? RL_MID_CTAS : 4)) * 128 / CH) k_main(RlDev D, RlBatch B, Src src, uint32_t weak) {
    using Smem = RlMainSmem<CELLS, CH>;
    constexpr int GT = Smem::GT;
    constexpr int PW = Smem::PW;
    extern __shared__ __align__(16) unsigned char rl_smem_raw[];
    Smem& sm = *reinterpret_cast<Smem*>(rl_smem_raw);
    uint32_t* const sm_t_pfx = reinterpret_cast<uint32_t*>(rl_smem_raw + sizeof(Smem));
    uint32_t* const sm_t_loc = sm_t_pfx + B.num_tiles + 1;

    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr bool lc = LC;  // load_counters: compile-time, so the default kernel carries none of it
    const bool write_out = (B.phase == RL_PHASE_COMMIT);
    const bool snapshot = Src::kCanBeMulti && (B.phase == RL_PHASE_SNAPSHOT);

    if (blockIdx.x == 0 && tid == 0) rl_trace(D.trace, D.trace_pos, RL_EV_MAIN, 0, D.seq);
    const uint32_t n_items = *B.n_items;
    const uint32_t ntile = B.num_tiles;
    const uint32_t tsz = rl_tile_of(B, rl_batch_n(B));
    for (;;) {
        // ---- next work item: atomic ticket, broadcast through shared memory -----------------------
        __syncthreads();  // the previous item is finished by every thread (sm.item is reused)
        if (tid == 0) sm.item = atomicAdd(B.ticket, 1u);
        for (uint32_t i = tid; i < GT; i += CH) sm.g_row[i] = 0xFFFFFFFFu;
        for (uint32_t i = tid; i < GT * PW; i += CH) sm.g_packed[i] = 0ull;
        __syncthreads();
        const uint32_t item = sm.item;
        if (item >= n_items) {
            // the last CTA to leave re-arms the ticket for the next launch over this workspace
            if (tid == 0 && atomicAdd(B.exit_ctr, 1u) == gridDim.x - 1) {
                *B.exit_ctr = 0;
                *B.ticket = 0;
                rl_trace(D.trace, D.trace_pos, RL_EV_MAIN, 1, D.seq);
            }
            break;
        }
        long long tph = D.kstats != nullptr ? clock64() : 0;
        const uint4 it = B.items[item];
        const uint32_t lo = it.y, hi = it.z;  // [lo, hi) of the partition's list
        // ---- the partition's list = its runs in the tiles' slices, tile after tile: merge on read --------
        {
            const uint32_t TL = B.nparts + B.nhot + 2;
            uint32_t carry = 0;
            for (uint32_t base = 0; base < ntile; base += CH) {  // CH tiles at a time: one pass for batches up to CH tiles
                const uint32_t t = base + tid;
                uint32_t c = 0;
                if (t < ntile) {
                    const uint32_t l0 = __ldcg(&B.tile_loc[(size_t)t * TL + it.x]);
                    const uint32_t l1 = __ldcg(&B.tile_loc[(size_t)t * TL + it.x + 1]);
                    c = l1 - l0;
                    sm_t_loc[t] = t * tsz + l0;
                }
                uint32_t x = c;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const uint32_t y = __shfl_up_sync(0xffffffffu, x, o);
                    if ((int)lane >= o) x += y;
                }
                if (lane == 31) sm.scan_w[warp] = x;
                __syncthreads();
                uint32_t woff = 0, tot = 0;
                for (uint32_t w = 0; w < (uint32_t)Smem::NW; w++) {
                    if (w < warp) woff += sm.scan_w[w];
                    tot += sm.scan_w[w];
                }
                if (t < ntile) sm_t_pfx[t] = carry + woff + x - c;
                carry += tot;
                __syncthreads();
            }
            if (tid == 0) sm_t_pfx[ntile] = carry;
            __syncthreads();
        }
        // position v of the list -> index into part_idx/part_row: the last tile whose prefix is <= v
        auto list_at = [&](uint32_t v) -> uint32_t {
            uint32_t a0 = 0, a1 = ntile - 1;
            while (a0 < a1) {
                const uint32_t mid = (a0 + a1 + 1) >> 1;
                if (sm_t_pfx[mid] <= v) a0 = mid;
                else a1 = mid - 1;
            }
            return sm_t_loc[a0] + (v - sm_t_pfx[a0]);
        };
        // Heavy partition: this CTA owns ONE chunk and the partition's chunks run concurrently under
        // optimistic concurrency control, row by row.  A chunk replays its requests against the
        // rows as they are (no row is written) and publishes the rows it read, each tagged with
        // whether its replay changes it.  Requests of different keys never interact, so a row's
        // history inside the batch is the sequence of chunks that touch it.  A row is "ordered"
        // for this chunk if an earlier chunk writes it (my read may be stale) or if I write it (an
        // earlier chunk may still have to read it).  With no ordered row the state this chunk saw
        // is the one sequential execution shows it and nobody before it can be disturbed by its
        // writes (a saturated hot key is read by every chunk and written by none): it commits at
        // once.  Otherwise it waits for exactly the earlier chunks touching an ordered row,
        // re-reads its rows and replays the keys whose state changed.  Earlier chunks hold lower
        // tickets, so they are running (or done) whenever a chunk waits for them.
        const bool chained = (it.w != RL_NONE_U32);
        // (access, row) pairs of the first chunk
        uint32_t na = 0, nrow = 0xFFFFFFFFu, npos = 0;
        if (lo + tid < hi) {
            npos = list_at(lo + tid);
            na = __ldcs(B.part_idx + npos);
            nrow = __ldcs(B.part_row + npos);
        }

        for (uint32_t c0 = lo; c0 < hi; c0 += CH) {
            // ---- 1. my access: gather the record, group by row while it is in flight --------------
            const uint32_t p = c0 + tid;
            const uint32_t a = na, myrow = nrow, mypos = npos;
            const bool valid = (p < hi) && (myrow != 0xFFFFFFFFu);  // no row: the region is full (error flagged by the probe)
            RlRaw rawrec;
            rawrec.w0 = make_ulonglong2(0ull, 0ull);
            rawrec.w1 = make_ulonglong2(0ull, 0ull);
            if (valid) rawrec = src.raw(a);
            if (p + CH < hi) {
                npos = list_at(p + CH);
                na = __ldcs(B.part_idx + npos);
                nrow = __ldcs(B.part_row + npos);
            }
            uint32_t slot = 0, gid = tid;
            bool is_rep = false;
            // lanes of a warp that hit the same row insert once (a hot row would otherwise serialise 32
            // same-address CAS per warp): `peers` = my row's lanes in this warp, kept for the ordinals and
            // for the warp-aggregated minima of the replay rounds
            const unsigned vmask = __ballot_sync(0xffffffffu, valid);
            unsigned peers = 0;
            int leader = 0;
            if (valid) {
                peers = __match_any_sync(vmask, myrow);
                leader = __ffs(peers) - 1;
                uint32_t s = 0;
                if ((int)lane == leader) {
                    s = rl_group_slot<GT>(myrow, weak);
                    for (;;) {
                        const uint32_t old = atomicCAS(&sm.g_row[s], 0xFFFFFFFFu, myrow);
                        if (old == 0xFFFFFFFFu) {
                            sm.g_rep[s] = tid;  // I claimed the slot: my row's group is mine to stage
                            is_rep = true;
                            break;
                        }
                        if (old == myrow) break;
                        s = (s + 1) & (GT - 1);
                    }
                }
                slot = __shfl_sync(peers, s, leader);
            }
            uint8_t* row = nullptr;
            RlRow<CELLS> st;
            if (is_rep) {
                // the row was located (or claimed) by the probe; its sectors are often still in L2
                row = D.rows + (size_t)myrow * RlGeom<GEO>::ROW_BYTES;
                rl_row_load<CELLS>(row, CELLS, st);
            }
            __syncthreads();
            if (valid) gid = sm.g_rep[slot];

            // ---- decode the record: limits of the cells I touch -----------------------------------
            RlReq acc;
            acc.req = 0; acc.cells = 0; acc.group = 0; acc.posorig = 0; acc.delta = 0; acc.now = 0;
            if (valid) src.decode(D, a, rawrec, acc);
            const uint64_t delta = acc.delta, now = acc.now;
            const RlCellDesc* gdesc = D.desc + (size_t)acc.group * 8;
            const uint32_t ncell = rl_cells_n(acc.cells);
            const bool multi = Src::kCanBeMulti && (MODE == 0) && rl_cells_multi(acc.cells);  // coupled to other rows
            RlMyLimits L;
            L.qmask = 0;
            constexpr bool kGeneric = LC || Src::kCanBeMulti;
            RlCellDesc mydesc[kGeneric ? CELLS : 1];  // generic variants: the limits of the cells I touch,
                                                      // indexed by cell, in local memory (L1) for the walks
#pragma unroll
            for (int k = 0; k < CELLS; k++) {
                L.mx[k] = 0;
                if (valid && (uint32_t)k < ncell) {
                    const uint32_t c = rl_cells_at(acc.cells, k);
                    const RlCellDesc d = gdesc[c];
                    if (kGeneric) mydesc[kGeneric ? c : 0] = d;
                    L.mx[k] = d.max_value;
                    L.qmask |= (d.qualified ? 1u : 0u) << k;
                }
            }
            const RlCellDesc* desc = kGeneric ? mydesc : gdesc;
            sm.d_arr[tid] = delta;
            sm.cells_arr[tid] = acc.cells;
            sm.g_flags[tid] = 0;
            sm.g_dirty[tid] = 0;
            sm.g_min[0][0][tid] = sm.g_min[0][1][tid] = 0xFFFFFFFFu;
            sm.g_min[1][0][tid] = sm.g_min[1][1][tid] = 0xFFFFFFFFu;
            RL_PHASE_TICK(0)  // item fetch + gather + grouping

            // ---- 2. stable ordinal: one packed add per (warp, row), one barrier --------------------
            if (valid && (int)lane == leader)
                atomicAdd(&sm.g_packed[slot * PW + (warp >> 3)], (unsigned long long)__popc(peers) << (8 * (warp & 7)));
            const bool solo = (peers & (peers - 1)) == 0;  // my row's only lane in this warp
            // ---- 3. the rep stages the row state -----------------------------------------------------
            if (is_rep) {
#pragma unroll
                for (int c = 0; c < CELLS; c++) {
                    sm.s_val[tid * CELLS + c] = st.value[c];
                    sm.s_exp[tid * CELLS + c] = st.expiry[c];
                }
                if (snapshot) {
                    B.log_row[mypos] = row;
#pragma unroll
                    for (int c = 0; c < CELLS; c++)
                        B.log_state[(size_t)mypos * GEO + c] = make_ulonglong2(st.value[c], st.expiry[c]);
                }
            }
            __syncthreads();
            uint32_t ord = 0, cnt = 0;
            if (valid) {
#pragma unroll
                for (int w = 0; w < Smem::NW; w++) {
                    const uint32_t f = (uint32_t)(sm.g_packed[slot * PW + (w >> 3)] >> (8 * (w & 7))) & 0xFFu;
                    cnt += f;
                    if ((uint32_t)w < warp) ord += f;
                }
                ord += __popc(peers & ((1u << lane) - 1));
            }
            // a row that dominates this chunk is a candidate for a partition of its own in the coming batches
            if (is_rep && B.nhot && cnt >= RL_HOT_MIN) {
                const uint32_t k = atomicAdd(D.hot_cand_n, 1u);
                if (k < RL_HOT_CAND) D.hot_cand[k] = myrow;
            }
            // a run of allowed requests is closed-form only over members that carry the rep's delta and
            // cell list: a member that differs is never part of a run (it ends the run before it and is
            // applied alone), so the members of any run are mutually alike
            const bool like_rep = valid && sm.d_arr[gid] == delta && sm.cells_arr[gid] == acc.cells;
            RL_PHASE_TICK(2)  // ordinals + row state staged

            // ---- 4. lock-step run-length replay -----------------------------------------------------
            bool done = !valid || snapshot;
            uint32_t pos = 0;
            for (int attempt = 0;; attempt++) {
            const uint32_t nrounds = rl_replay_rounds<CELLS, MODE, LC>(
                B, write_out, &sm.s_val[gid * CELLS], &sm.s_exp[gid * CELLS], &sm.g_min[0][0][gid], CH, &sm.g_dirty[gid], acc, L,
                desc, gdesc, multi, like_rep, valid, peers, solo, leader, lane, ord, cnt, done, pos);
            if (tid == 0) {
                RL_KSTAT_ADD(0, 1);
                RL_KSTAT_ADD(1, nrounds);
            }
            RL_PHASE_TICK(3)  // replay rounds
            if (!chained || snapshot || attempt == 1) break;
            if (tid == 0) RL_KSTAT_ADD(2, 1);
            const uint32_t base_item = item - it.w;  // first chunk of my partition
            // (b) publish the rows I touched, each tagged with "I write it" (under my speculation);
            //     the grouping table g_row IS the set of rows this chunk read
            for (uint32_t i = tid; i < GT; i += CH) sm.rflag[i] = 0;
            for (uint32_t i = tid; i < 64; i += CH) sm.need_bits[i] = 0;
            if (tid == 0) sm.w_cnt = 0;
            __syncthreads();
            if (is_rep) {
                // a row I WRITE is ordered too: no earlier chunk may still be reading it when I commit
                if (sm.g_dirty[tid]) sm.rflag[slot] = 1;
                B.chain_w[(size_t)item * CH + atomicAdd(&sm.w_cnt, 1u)] = (myrow << 1) | (sm.g_dirty[tid] ? 1u : 0u);
                __threadfence();  // my entry is visible device-wide before the status word says so
            }
            __syncthreads();
            if (tid == 0) {
                B.chain_wcnt[item] = sm.w_cnt;
                __threadfence();
                atomicExch(B.chain_status + item, 1u);
            }
            // (c) wait until every earlier chunk of the partition has published its set
            for (;;) {
                bool ok = true;
                for (uint32_t j = tid; j < it.w; j += CH)
                    ok = ok && (*(volatile uint32_t*)(B.chain_status + base_item + j) >= 1u);
                if (__syncthreads_and(ok)) break;
                __nanosleep(RL_WAIT_NS);
            }
            __threadfence();
            // (d) rows I read that some earlier chunk writes: their history must be replayed in order.
            //     Pass 1 flags those rows, pass 2 collects every earlier chunk that touches one of them
            //     (a chunk that only READS such a row may turn into a writer once it re-validates).
            //     The earlier chunks' sets are scanned CH chunks at a time, flattened: thread t fetches
            //     the size of chunk blk*CH+t, a block scan turns sizes into offsets, and the threads then
            //     stride over all the entries of those chunks at once (independent loads, not one
            //     dependent round trip per earlier chunk).
            bool any_dep = false;
            for (int pass = 0; pass < 2; pass++) {
                bool flagged = is_rep && sm.g_dirty[tid] != 0;
                for (uint32_t blk = 0; blk < it.w; blk += CH) {
                    const uint32_t jn = min((uint32_t)CH, it.w - blk);  // chunks in this block
                    const uint32_t myc = (tid < jn) ? __ldcg(B.chain_wcnt + base_item + blk + tid) : 0;
                    uint32_t x = myc;
#pragma unroll
                    for (int o = 1; o < 32; o <<= 1) {
                        const uint32_t y = __shfl_up_sync(0xffffffffu, x, o);
                        if ((int)lane >= o) x += y;
                    }
                    if (lane == 31) sm.scan_w[warp] = x;
                    __syncthreads();
                    uint32_t woff = 0, total = 0;
                    for (uint32_t w = 0; w < Smem::NW; w++) {
                        if (w < warp) woff += sm.scan_w[w];
                        total += sm.scan_w[w];
                    }
                    sm.scan_off[tid] = woff + x - myc;  // exclusive offset of chunk blk+tid
                    __syncthreads();
                    for (uint32_t q = tid; q < total; q += CH) {
                        // chunk holding flattened entry q: last j with scan_off[j] <= q
                        uint32_t blo = 0, bhi = jn - 1;
                        while (blo < bhi) {
                            const uint32_t mid = (blo + bhi + 1) >> 1;
                            if (sm.scan_off[mid] <= q) blo = mid;
                            else bhi = mid - 1;
                        }
                        const uint32_t j = blk + blo;
                        const uint32_t e = __ldcg(B.chain_w + (size_t)(base_item + j) * CH + (q - sm.scan_off[blo]));
                        const uint32_t w = e >> 1;
                        uint32_t s2 = rl_group_slot<GT>(w, weak);
                        for (;;) {
                            const uint32_t xs = sm.g_row[s2];
                            if (xs == w) {
                                if (pass == 0) {
                                    if (e & 1u) {
                                        sm.rflag[s2] = 1;
                                        flagged = true;
                                    }
                                } else if (sm.rflag[s2]) {
                                    any_dep = true;
                                    atomicOr(&sm.need_bits[(j >> 5) & 63], (j < 2048) ? (1u << (j & 31)) : 0u);
                                }
                                break;
                            }
                            if (xs == 0xFFFFFFFFu) break;
                            s2 = (s2 + 1) & (GT - 1);
                        }
                    }
                    __syncthreads();  // scan_off / scan_w are reused by the next block
                }
                if (pass == 0) {
                    if (!__syncthreads_or(flagged)) break;  // no ordered row
                } else {
                    any_dep = __syncthreads_or(any_dep);
                }
            }
            if (!any_dep) break;  // nothing I read is written before me: commit now, in parallel
            if (tid == 0) RL_KSTAT_ADD(3, 1);
            // (e) wait for the chunks my rows depend on to commit, then re-validate
            for (;;) {
                bool ok = true;
                for (uint32_t j = tid; j < it.w; j += CH) {
                    const bool need = (j >= 2048) || ((sm.need_bits[j >> 5] >> (j & 31)) & 1u);
                    if (need) ok = ok && (*(volatile uint32_t*)(B.chain_status + base_item + j) == 4u);
                }
                if (__syncthreads_and(ok)) break;
                __nanosleep(RL_WAIT_NS);
            }
            __threadfence();
            bool redo = false;
            if (is_rep) {
                RlRow<CELLS> cur;
                rl_row_load<CELLS>(row, CELLS, cur);
                bool same = true;
#pragma unroll
                for (int c = 0; c < CELLS; c++) same = same && cur.value[c] == st.value[c] && cur.expiry[c] == st.expiry[c];
                if (!same) {  // an earlier chunk changed this key: replay it from the committed state
                    st = cur;
#pragma unroll
                    for (int c = 0; c < CELLS; c++) {
                        sm.s_val[tid * CELLS + c] = cur.value[c];
                        sm.s_exp[tid * CELLS + c] = cur.expiry[c];
                    }
                    sm.g_dirty[tid] = 0;
                    sm.g_min[0][0][tid] = sm.g_min[0][1][tid] = 0xFFFFFFFFu;
                    sm.g_min[1][0][tid] = sm.g_min[1][1][tid] = 0xFFFFFFFFu;
                    sm.g_flags[tid] |= 4u;
                    redo = true;
                }
            }
            if (!__syncthreads_or(redo)) break;
            if (valid && (sm.g_flags[gid] & 4u)) {
                done = false;
                pos = 0;
            }
            }

            RL_PHASE_TICK(4)  // optimistic-commit protocol (chained chunks)
            // ---- 5. write the dirty cells back -------------------------------------------------------
            if (is_rep && !snapshot) {
                const uint32_t dirty = sm.g_dirty[tid];
#pragma unroll
                for (int c = 0; c < CELLS; c++)
                    if (dirty & (1u << c))
                        rl_st_cg(row + 16 + 16 * c, sm.s_val[tid * CELLS + c], sm.s_exp[tid * CELLS + c]);
                if (chained && dirty) __threadfence();
            }
            __syncthreads();
            if (chained && !snapshot && tid == 0) atomicExch(B.chain_status + item, 4u);
            // grouping tables of the next chunk of this item
            if (c0 + CH < hi) {
                for (uint32_t i = tid; i < GT; i += CH) sm.g_row[i] = 0xFFFFFFFFu;
                for (uint32_t i = tid; i < GT * PW; i += CH) sm.g_packed[i] = 0ull;
                __syncthreads();
            }
            RL_PHASE_TICK(5)  // write-back
        }
    }
}

// ---------------------------------------------------------------------------------------
// Hot rows.  CTA h replays the whole request list of hot slot h (partition nparts + h: ONE table row) in
// stream order.  Same exact run-length logic as k_main (DESIGN.md §3.3) — but a "round" here SWEEPS the whole
// remaining list (up to RL_HOT_SWEEP requests), not one chunk: from position `pos` with row state S,
//   A  the longest prefix of requests denied under S without any effect is final as it stands;
//   B  the longest prefix of requests that look like the one at `pos` (delta, cells) and are all allowed
//      without a window reset or insert: request i sees S plus (i - pos) deltas — closed form;
//   else the request at `pos` is applied alone with the sequential rule.
// Pass 1 of a sweep finds the two prefix lengths (every thread strides over the list and keeps the first
// position where A / B fails; one CTA-wide minimum, one barrier for the whole list); pass 2 writes the
// verdicts of the prefix that won.  A saturated row (all denied) or a row far from its limit (all allowed)
// costs ONE sweep whatever its length — 6 500 requests of C2's hottest key in a few microseconds — and a
// window rollover three.  There is nothing to group and nothing to chain: the row state lives in shared
// memory from the first request of the batch to the last.  This is what stands in for "warp-aggregated
// atomics" in the hot-key case (BASELINE.json configs[4]): atomics would hand out allow/deny by arrival order.
#ifndef RL_HOT_SWEEP
#define RL_HOT_SWEEP (64 * RL_HOT_THREADS)  // requests one sweep looks at (bounds the work thrown away by a short prefix)
#endif
template <int GEO, int CELLS, class Src, int MODE, bool LC>
__global__ void __launch_bounds__(RL_HOT_THREADS) k_hot(RlDev D, RlBatch B, Src src) {
    constexpr int CH = RL_HOT_THREADS;
    __shared__ uint32_t t_pfx[RL_MAX_TILES + 1], t_loc[RL_MAX_TILES], scan_w[CH / 32];
    __shared__ unsigned long long s_val[CELLS], s_exp[CELLS];
    __shared__ RlCellDesc s_desc[8];  // the row group's limits
    __shared__ RlReq s_head;          // the request at `pos`
    __shared__ uint32_t s_min[2], s_dirty;
    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t q = B.nparts + blockIdx.x;
    const uint32_t ntile = B.num_tiles;
    const uint32_t tsz = rl_tile_of(B, rl_batch_n(B));
    const uint32_t TL = B.nparts + B.nhot + 2;
    {
        uint32_t carry = 0;
        for (uint32_t base = 0; base < ntile; base += CH) {
            const uint32_t t = base + tid;
            uint32_t c = 0;
            if (t < ntile) {
                const uint32_t l0 = __ldcg(&B.tile_loc[(size_t)t * TL + q]);
                const uint32_t l1 = __ldcg(&B.tile_loc[(size_t)t * TL + q + 1]);
                c = l1 - l0;
                t_loc[t] = t * tsz + l0;
            }
            uint32_t x = c;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t y = __shfl_up_sync(0xffffffffu, x, o);
                if ((int)lane >= o) x += y;
            }
            if (lane == 31) scan_w[warp] = x;
            __syncthreads();
            uint32_t woff = 0, tot = 0;
            for (uint32_t w = 0; w < CH / 32; w++) {
                if (w < warp) woff += scan_w[w];
                tot += scan_w[w];
            }
            if (t < ntile) t_pfx[t] = carry + woff + x - c;
            carry += tot;
            __syncthreads();
        }
        if (tid == 0) t_pfx[ntile] = carry;
        __syncthreads();
    }
    const uint32_t total = t_pfx[ntile];
    if (total == 0) return;
    if (tid == 0) rl_trace(D.trace, D.trace_pos, RL_EV_HOT, 0, total);  // per hot row: list length, start .. end
    auto list_at = [&](uint32_t v) -> uint32_t {
        uint32_t a0 = 0, a1 = ntile - 1;
        while (a0 < a1) {
            const uint32_t mid = (a0 + a1 + 1) >> 1;
            if (t_pfx[mid] <= v) a0 = mid;
            else a1 = mid - 1;
        }
        return t_loc[a0] + (v - t_pfx[a0]);
    };
    // request i of the list, decoded
    auto fetch = [&](uint32_t i, RlReq& acc) {
        const uint32_t a = __ldcs(B.part_idx + list_at(i));
        const RlRaw w = src.raw(a);
        src.decode(D, a, w, acc);
    };
    const uint32_t rowidx = __ldcg(B.part_row + list_at(0));
    uint8_t* row = D.rows + (size_t)rowidx * RlGeom<GEO>::ROW_BYTES;
    if (tid < CELLS) {
        const ulonglong2 v = rl_ld_cg(row + 16 + 16 * tid);
        s_val[tid] = v.x;
        s_exp[tid] = v.y;
    }
    if (tid == 0) {
        s_dirty = 0;
        fetch(0, s_head);
    }
    __syncthreads();
    if (tid < 8) s_desc[tid] = D.desc[(size_t)s_head.group * 8 + tid];  // one row => one row group
    __syncthreads();

    // limits of the cells request `acc` touches, in its own cell order (shared-memory copies)
    auto limits_of = [&](const RlReq& acc, RlMyLimits& L) {
        const uint32_t n = rl_cells_n(acc.cells);
        L.qmask = 0;
#pragma unroll
        for (int k = 0; k < CELLS; k++) {
            L.mx[k] = 0;
            if ((uint32_t)k < n) {
                const uint32_t c = rl_cells_at(acc.cells, k);
                L.mx[k] = s_desc[c].max_value;
                L.qmask |= (s_desc[c].qualified ? 1u : 0u) << k;
            }
        }
    };
    auto write_first = [&](const RlReq& acc, uint32_t fl) {
        if (!B.out_first_limited) return;
        if (fl == RL_NONE_U32) {
            B.out_first_limited[acc.req] = RL_NONE_U32;
            return;
        }
        const uint32_t n = rl_cells_n(acc.cells);
#pragma unroll
        for (int k = 0; k < CELLS; k++)
            if ((uint32_t)k < n && rl_pos_at(acc.posorig, k) == fl) B.out_first_limited[acc.req] = s_desc[rl_cells_at(acc.cells, k)].limit_id;
    };
    auto lc_outputs = [&](const RlReq& acc, uint64_t*& rem, uint64_t*& ttl) {
        rem = ttl = nullptr;
        if (MODE == 0 && LC) {
            const size_t ob = B.out_off ? (size_t)B.out_off[acc.req] : (size_t)acc.req * B.out_stride;
            if (B.out_remaining) rem = B.out_remaining + ob;
            if (B.out_ttl) ttl = B.out_ttl + ob;
        }
    };

    uint32_t pos = 0;
    while (pos < total) {
        // ---- pass 1: how far do hypotheses A and B hold from `pos` under the state S? -------------------
        const uint32_t end = min(total, pos + (uint32_t)RL_HOT_SWEEP);
        RlRow<CELLS> S;
#pragma unroll
        for (int c = 0; c < CELLS; c++) {
            S.value[c] = s_val[c];
            S.expiry[c] = s_exp[c];
        }
        const RlReq head = s_head;
        if (tid == 0) s_min[0] = s_min[1] = end;
        __syncthreads();
        uint32_t fa = end, fb = end;  // first position where A / B fails, among mine
        constexpr int U = 4;          // strides in flight per thread: index and record loads of U requests overlap
        for (uint32_t i0 = pos + tid; i0 < end && (fa == end || fb == end); i0 += CH * U) {
            uint32_t ai[U];
            RlRaw wi[U];
#pragma unroll
            for (int u = 0; u < U; u++) {
                const uint32_t i = i0 + u * CH;
                ai[u] = (i < end) ? __ldcs(B.part_idx + list_at(i)) : 0u;
            }
#pragma unroll
            for (int u = 0; u < U; u++)
                if (i0 + u * CH < end) wi[u] = src.raw(ai[u]);
#pragma unroll
            for (int u = 0; u < U; u++) {
                const uint32_t i = i0 + u * CH;
                if (i >= end) break;
                RlReq acc;
                src.decode(D, ai[u], wi[u], acc);
                RlMyLimits L;
                limits_of(acc, L);
                bool aok, bok;
                uint32_t fl;
                rl_eval_ab<CELLS>((const unsigned long long*)S.value, (const unsigned long long*)S.expiry, L, acc.cells, acc.posorig, acc.delta,
                                  (uint64_t)(i - pos + 1) * acc.delta, acc.now, LC, MODE == 0, aok, bok, fl);
                if (MODE == 2) aok = false;
                bok = bok && acc.delta == head.delta && acc.cells == head.cells;
                if (!aok && fa == end) fa = i;
                if (!bok && fb == end) fb = i;
            }
        }
        fa = __reduce_min_sync(0xffffffffu, fa);
        fb = __reduce_min_sync(0xffffffffu, fb);
        if (lane == 0) {
            if (fa < end) atomicMin(&s_min[0], fa);
            if (fb < end) atomicMin(&s_min[1], fb);
        }
        __syncthreads();
        const uint32_t mA = s_min[0], mB = s_min[1];
        uint32_t newpos;
        // ---- pass 2: the prefix that won is final -------------------------------------------------------
        if (mA > pos) {  // denied under S, nothing changes
            newpos = mA;
            for (uint32_t i0 = pos + tid; i0 < newpos; i0 += CH * U) {
                uint32_t ai[U];
                RlRaw wi[U];
#pragma unroll
                for (int u = 0; u < U; u++) ai[u] = (i0 + u * CH < newpos) ? __ldcs(B.part_idx + list_at(i0 + u * CH)) : 0u;
#pragma unroll
                for (int u = 0; u < U; u++)
                    if (i0 + u * CH < newpos) wi[u] = src.raw(ai[u]);
#pragma unroll
                for (int u = 0; u < U; u++) {
                if (i0 + u * CH >= newpos) break;
                RlReq acc;
                src.decode(D, ai[u], wi[u], acc);
                uint32_t fl;
                if (LC) {
                    RlRow<CELLS> loc = S;
                    uint32_t dirty = 0;
                    uint64_t *rem, *ttl;
                    lc_outputs(acc, rem, ttl);
                    fl = rl_walk_check_single<CELLS>(loc, dirty, s_desc, acc.cells, acc.posorig, acc.delta, acc.now, true, rem, ttl);
                } else {
                    RlMyLimits L;
                    limits_of(acc, L);
                    bool aok, bok;
                    rl_eval_ab<CELLS>((const unsigned long long*)S.value, (const unsigned long long*)S.expiry, L, acc.cells, acc.posorig, acc.delta,
                                      acc.delta, acc.now, false, true, aok, bok, fl);
                }
                rl_store_verdict(B, acc.req, 1);
                write_first(acc, fl);
                }
            }
        } else if (mB > pos) {  // allowed, values accumulate: request i sees S + (i - pos) deltas
            newpos = mB;
            if (MODE == 0) {
                for (uint32_t i0 = pos + tid; i0 < newpos; i0 += CH * U) {
                    uint32_t ai[U];
                    RlRaw wi[U];
#pragma unroll
                    for (int u = 0; u < U; u++) ai[u] = (i0 + u * CH < newpos) ? __ldcs(B.part_idx + list_at(i0 + u * CH)) : 0u;
#pragma unroll
                    for (int u = 0; u < U; u++)
                        if (i0 + u * CH < newpos) wi[u] = src.raw(ai[u]);
#pragma unroll
                    for (int u = 0; u < U; u++) {
                    const uint32_t i = i0 + u * CH;
                    if (i >= newpos) break;
                    RlReq acc;
                    src.decode(D, ai[u], wi[u], acc);
                    if (LC) {
                        RlRow<CELLS> loc = S;
                        rl_advance_run<CELLS>(loc, acc.cells, (uint64_t)(i - pos) * acc.delta);
                        uint32_t dirty = 0;
                        uint64_t *rem, *ttl;
                        lc_outputs(acc, rem, ttl);
                        rl_walk_check_single<CELLS>(loc, dirty, s_desc, acc.cells, acc.posorig, acc.delta, acc.now, true, rem, ttl);
                    }
                    rl_store_verdict(B, acc.req, 0);
                    write_first(acc, RL_NONE_U32);
                    }
                }
            }
            if (tid == 0) {
                const uint64_t add = (uint64_t)(newpos - pos) * head.delta;
                const uint32_t n = rl_cells_n(head.cells);
                uint32_t dirty = 0;
                for (uint32_t k = 0; k < n; k++) {
                    const uint32_t c = rl_cells_at(head.cells, k);
                    s_val[c] += add;
                    dirty |= 1u << c;
                }
                s_dirty |= dirty;
            }
        } else {  // the request at `pos`, alone, by the sequential rule (rl_core.h)
            newpos = pos + 1;
            if (tid == 0) {
                RlRow<CELLS> loc = S;
                uint32_t dirty = 0, fl = RL_NONE_U32;
                uint64_t *rem, *ttl;
                lc_outputs(head, rem, ttl);
                if (MODE == 2) rl_walk_update<CELLS>(loc, dirty, s_desc, head.cells, head.delta, head.now);
                else fl = rl_walk_check_single<CELLS>(loc, dirty, s_desc, head.cells, head.posorig, head.delta, head.now, LC, rem, ttl);
#pragma unroll
                for (int c = 0; c < CELLS; c++)
                    if (dirty & (1u << c)) {
                        s_val[c] = loc.value[c];
                        s_exp[c] = loc.expiry[c];
                    }
                s_dirty |= dirty;
                if (MODE == 0) {
                    rl_store_verdict(B, head.req, (uint8_t)(fl != RL_NONE_U32));
                    write_first(head, fl);
                }
            }
        }
        pos = newpos;
        __syncthreads();  // every read of S / s_head / s_min of this sweep is done
        if (tid == 0 && pos < total) fetch(pos, s_head);
        __syncthreads();
    }
    if (tid < CELLS && ((s_dirty >> tid) & 1u)) rl_st_cg(row + 16 + 16 * tid, s_val[tid], s_exp[tid]);
    if (tid == 0) rl_trace(D.trace, D.trace_pos, RL_EV_HOT, 1, total);
}

// ---------------------------------------------------------------------------------------
// Resolve kernels: request -> accesses (rl_resolve_request in rl_core.h).
struct RlResolveOut {
    RlAccess* acc;
    uint64_t* delta;  // records only: materialised per request
    uint64_t* now;
    uint8_t* out_limited;         // defaults for requests without counters
    uint32_t* out_first_limited;  // nullable
};

__global__ void k_resolve_csr(RlDev D, uint32_t n, const uint32_t* __restrict__ off,
                              const rl_counter* __restrict__ ctrs, const uint64_t* __restrict__ now, RlResolveOut O,
                              int write_defaults) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t o0 = off[i], m = off[i + 1] - o0;
    if (m == 0) {
        if (write_defaults) {
            O.out_limited[i] = 0;
            if (O.out_first_limited) O.out_first_limited[i] = RL_NONE_U32;
        }
        return;
    }
    auto get = [&](uint32_t j) {
        const rl_counter c = ctrs[o0 + j];
        RlCtrIn r;
        r.limit_id = c.limit_id;
        r.key_lo = c.key_lo;
        r.key_hi = c.key_hi;
        return r;
    };
    RlAccess tmp[RL_MAX_CTRS_PER_REQ];
    const int nacc = now[i] == 0 ? -(int)RL_DEV_CLOCK : rl_resolve_request(i, m, get, D.limits, D.limits_cap, true, tmp);
    if (nacc < 0) {
        rl_set_err(D, (uint32_t)(-nacc));
        for (uint32_t x = 0; x < m && x < RL_MAX_CTRS_PER_REQ; x++) {
            RlAccess z;
            z.key_lo = 0;
            z.hdr_hi = 0;
            z.req = i;
            z.cells = 0;
            z.posorig = 0;
            O.acc[o0 + x] = z;
        }
        // slots beyond RL_MAX_CTRS_PER_REQ (too-many-counters error) are cleared too
        for (uint32_t x = RL_MAX_CTRS_PER_REQ; x < m; x++) {
            RlAccess z;
            z.key_lo = 0;
            z.hdr_hi = 0;
            z.req = i;
            z.cells = 0;
            z.posorig = 0;
            O.acc[o0 + x] = z;
        }
        if (write_defaults) O.out_limited[i] = 0;
        return;
    }
    for (uint32_t x = 0; x < m; x++) O.acc[o0 + x] = tmp[x];
    if (nacc > 1) atomicOr(D.flags, 1u);
}

// Records whose namespaces span several rows: slot base = i * stride.
__global__ void k_resolve_records(RlDev D, uint32_t n, const rl_record* __restrict__ recs, uint32_t stride,
                                  RlResolveOut O, int write_defaults) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const rl_record rec = recs[i];
    O.delta[i] = rec.hits_addend;
    O.now[i] = rec.now_us;
    uint32_t m = 0, lim_off = 0;
    if (rec.ns_id < D.ns_cap) {
        const RlNsDev ns = D.ns[rec.ns_id];
        m = ns.lim_cnt;
        lim_off = ns.lim_off;
    }
    const size_t o0 = (size_t)i * stride;
    RlAccess z;
    z.key_lo = 0;
    z.hdr_hi = 0;
    z.req = i;
    z.cells = 0;
    z.posorig = 0;
    if (m == 0) {
        for (uint32_t x = 0; x < stride; x++) O.acc[o0 + x] = z;
        if (write_defaults) {
            O.out_limited[i] = 0;
            if (O.out_first_limited) O.out_first_limited[i] = RL_NONE_U32;
        }
        return;
    }
    auto get = [&](uint32_t j) {
        RlCtrIn r;
        r.limit_id = D.ns_limit_ids[lim_off + j];
        r.key_lo = rec.key_lo;
        r.key_hi = rec.key_hi & RL_RECORD_KEY_HI_MASK;
        return r;
    };
    RlAccess tmp[RL_MAX_CTRS_PER_REQ];
    const int nacc =
        rec.now_us == 0 ? -(int)RL_DEV_CLOCK : rl_resolve_request(i, m, get, D.limits, D.limits_cap, true, tmp);
    if (nacc < 0) {
        rl_set_err(D, (uint32_t)(-nacc));
        for (uint32_t x = 0; x < stride; x++) O.acc[o0 + x] = z;
        if (write_defaults) O.out_limited[i] = 0;
        return;
    }
    for (uint32_t x = 0; x < stride; x++) O.acc[o0 + x] = (x < m) ? tmp[x] : z;
    if (nacc > 1) atomicOr(D.flags, 1u);
}

// Undo a speculative round: put every logged row back to its state at batch start.
template <int CELLS>
__global__ void k_restore(uint32_t n_acc, uint32_t act, uint8_t* const* __restrict__ log_row,
                          const ulonglong2* __restrict__ log_state) {
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n_acc) return;
    uint8_t* row = log_row[p];
    if (!row) return;
#pragma unroll
    for (int c = 0; c < CELLS; c++) {
        if ((uint32_t)c >= act) break;  // only the cells in use were logged
        const ulonglong2 v = log_state[(size_t)p * CELLS + c];
        rl_st_cg(row + 16 + 16 * c, v.x, v.y);
    }
}

// fixed-point bookkeeping: changed |= (prev != next); prev = next; next = NONE
__global__ void k_fl_step(uint32_t n, uint32_t* fl_prev, uint32_t* fl_next, uint32_t* changed) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t p = fl_prev[i], x = fl_next[i];
    if (p != x) {
        fl_prev[i] = x;
        atomicOr(changed, 1u);
    }
    fl_next[i] = RL_NONE_U32;
}

// ---------------------------------------------------------------------------------------
// is_rate_limited (lib.rs:362-409 over in_memory.rs:20-35): read-only, one thread per
// request, counters in the given order, no insert.
template <int CELLS>
__device__ __forceinline__ bool rl_query_counter(const RlDev& D, uint32_t limit_id, uint64_t key_lo,
                                                 uint64_t key_hi, uint64_t delta, uint64_t now, bool& err) {
    if (limit_id >= D.limits_cap || D.limits[limit_id].group == 0) {
        rl_set_err(D, RL_DEV_UNKNOWN_LIMIT);
        err = true;
        return false;
    }
    const RlLimitDev l = D.limits[limit_id];
    if (l.qualified && (key_hi >> 32)) {
        rl_set_err(D, RL_DEV_KEY_RANGE);
        err = true;
        return false;
    }
    const uint64_t klo = l.qualified ? key_lo : 0;
    const uint64_t hhi = ((uint64_t)l.group << 32) | (l.qualified ? key_hi : 0);
    const uint8_t* row = rl_probe<CELLS>(D, rl_row_hash(klo, hhi), klo, hhi, false);
    uint64_t v = 0;
    if (row) {
        const ulonglong2 c = rl_ld_cg(row + 16 + 16 * l.cell);
        v = rl_value_at(c.x, c.y, now);
    }
    const RlCellDesc d = D.desc[(size_t)l.group * 8 + l.cell];
    return !(d.max_value >= v + delta);  // in_memory.rs:34
}

template <int CELLS>
__global__ void k_query_csr(RlDev D, uint32_t n, const uint32_t* __restrict__ off,
                            const rl_counter* __restrict__ ctrs, const uint64_t* __restrict__ delta,
                            const uint64_t* __restrict__ now, uint8_t* out_limited, uint32_t* out_first) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t first = RL_NONE_U32;
    const uint64_t d = delta[i], t = now[i];
    for (uint32_t j = off[i]; j < off[i + 1]; j++) {
        const rl_counter c = ctrs[j];
        bool err = false;
        if (rl_query_counter<CELLS>(D, c.limit_id, c.key_lo, c.key_hi, d, t, err)) {
            first = c.limit_id;
            break;
        }
        if (err) break;
    }
    out_limited[i] = (first != RL_NONE_U32);
    if (out_first) out_first[i] = first;
}

template <int CELLS>
__global__ void k_query_records(RlDev D, uint32_t n, const rl_record* __restrict__ recs, uint8_t* out_limited,
                                uint32_t* out_first) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const rl_record rec = recs[i];
    uint32_t first = RL_NONE_U32;
    if (rec.ns_id < D.ns_cap) {
        const RlNsDev ns = D.ns[rec.ns_id];
        for (uint32_t j = 0; j < ns.lim_cnt; j++) {
            const uint32_t lid = D.ns_limit_ids[ns.lim_off + j];
            bool err = false;
            if (rl_query_counter<CELLS>(D, lid, rec.key_lo, rec.key_hi & RL_RECORD_KEY_HI_MASK, rec.hits_addend, rec.now_us, err)) {
                first = lid;
                break;
            }
            if (err) break;
        }
    }
    out_limited[i] = (first != RL_NONE_U32);
    if (out_first) out_first[i] = first;
}

// ---------------------------------------------------------------------------------------
// Maintenance kernels: streaming passes over the slab, one thread per row.
struct RlScanOut {
    uint32_t* limit_id;
    uint64_t* key_lo;
    uint64_t* key_hi;
    uint64_t* a;  // dump: value      | get_counters: remaining
    uint64_t* b;  // dump: expiry_us  | get_counters: ttl_us
    unsigned long long* count;
    uint64_t cap;
};

// mode 0: dump every present cell; mode 1: get_counters (ns_sel[ns]!=0, ttl>0)
template <int CELLS>
__global__ void k_scan(RlDev D, uint64_t nrows, int mode, uint64_t now, const uint8_t* __restrict__ ns_sel,
                       const uint32_t* __restrict__ group_ns, RlScanOut O) {
    constexpr uint32_t RB = RlGeom<CELLS>::ROW_BYTES;
    const uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= nrows) return;
    const uint8_t* row = D.rows + r * RB;
    const ulonglong2 hdr = rl_ld_cg(row);
    if (hdr.y == 0 || hdr.y == RL_TOMB_HI) return;
    const uint32_t group = (uint32_t)(hdr.y >> 32);
    if (mode == 1 && !ns_sel[group_ns[group]]) return;
    const RlCellDesc* desc = D.desc + (size_t)group * 8;
#pragma unroll
    for (int c = 0; c < CELLS; c++) {
        const RlCellDesc d = desc[c];
        if (d.limit_id == RL_NONE_U32) continue;
        const ulonglong2 cell = rl_ld_cg(row + 16 + 16 * c);
        if (d.qualified && cell.y == 0) continue;  // logically absent
        uint64_t a = cell.x, b = cell.y;
        if (mode == 1) {
            const uint64_t ttl = rl_ttl(cell.y, now);
            if (ttl == 0) continue;                               // in_memory.rs:167-169
            a = d.max_value - rl_value_at(cell.x, cell.y, now);   // wrapping, :164-165
            b = ttl;
        }
        const unsigned long long pos = atomicAdd(O.count, 1ull);
        if (pos < O.cap) {
            O.limit_id[pos] = d.limit_id;
            O.key_lo[pos] = hdr.x;
            O.key_hi[pos] = hdr.y & 0xFFFFFFFFull;
            O.a[pos] = a;
            O.b[pos] = b;
        }
    }
}

// delete_counters (in_memory.rs:241-257): reset the cells of the selected limits.
// sweep (mode 1): invalidate qualified cells with 0 < expiry <= now; rows left with no live
// cell and no unqualified cell become tombstones.
template <int CELLS>
__global__ void k_reset(RlDev D, uint64_t nrows, int mode, uint64_t now, const uint8_t* __restrict__ limit_sel,
                        unsigned long long* count) {
    constexpr uint32_t RB = RlGeom<CELLS>::ROW_BYTES;
    const uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= nrows) return;
    uint8_t* row = D.rows + r * RB;
    const ulonglong2 hdr = rl_ld_cg(row);
    if (hdr.y == 0 || hdr.y == RL_TOMB_HI) return;
    const uint32_t group = (uint32_t)(hdr.y >> 32);
    const RlCellDesc* desc = D.desc + (size_t)group * 8;
    bool any_live = false, any_unq = false;
    uint32_t dropped = 0;
#pragma unroll
    for (int c = 0; c < CELLS; c++) {
        const RlCellDesc d = desc[c];
        const ulonglong2 cell = rl_ld_cg(row + 16 + 16 * c);
        bool kill = false;
        if (mode == 0) {
            kill = d.limit_id != RL_NONE_U32 && limit_sel[d.limit_id] && (cell.x != 0 || cell.y != 0);
        } else {
            kill = d.limit_id != RL_NONE_U32 && d.qualified && cell.y != 0 && cell.y <= now;
        }
        if (kill) {
            rl_st_cg(row + 16 + 16 * c, 0ull, 0ull);
            dropped++;
        } else if (d.limit_id != RL_NONE_U32) {
            if (!d.qualified) any_unq = true;
            else if (cell.y != 0) any_live = true;
        } else if (cell.x != 0 || cell.y != 0) {
            rl_st_cg(row + 16 + 16 * c, 0ull, 0ull);  // cell of a forgotten limit
        }
    }
    if (mode == 1 && !any_live && !any_unq) rl_st_cg(row, 0ull, RL_TOMB_HI);
    if (dropped && count) atomicAdd(count, (unsigned long long)dropped);
}

// ---------------------------------------------------------------------------------------
// Multi-GPU exchange helpers: stable bucketing of records by owner rank (world <= 32).
// Same tile/warp-slice scheme as k_part, with the owner as the bucket.
__device__ __forceinline__ uint32_t rl_owner_dev(uint32_t ns_id, uint32_t world) {
    return (uint32_t)(rl_mix64((uint64_t)ns_id + 0x51ed270b0a1fULL) % world);
}

// slot_cap == 0: compact output (owner o's records at owner_base[o]...), out_src[pos] = a.
// slot_cap  > 0: fixed-size blocks (owner o's records at o*slot_cap..., at most slot_cap of them;
//                the caller pre-fills the buffer with no-op records), out_pos[a] = pos or ~0.
template <bool SCATTER>
__global__ void __launch_bounds__(RL_PART_THREADS) k_bucket(const rl_record* __restrict__ recs, uint32_t n,
                                                           uint32_t world, uint32_t tile, uint32_t* tile_cnt,
                                                           const uint32_t* __restrict__ owner_base,
                                                           rl_record* out_recs, uint32_t* out_src, uint32_t slot_cap,
                                                           uint32_t* out_pos) {
    __shared__ uint32_t wcnt[RL_PART_WARPS][32];
    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t t0 = blockIdx.x * tile, t1 = min(t0 + tile, n);
    const uint32_t slice = tile / RL_PART_WARPS;
    const uint32_t s0 = min(t0 + warp * slice, t1), s1 = min(s0 + slice, t1);
    wcnt[warp][lane] = 0;
    __syncthreads();
    for (uint32_t b = s0; b < s1; b += 32) {
        const uint32_t a = b + lane;
        const bool valid = a < s1;
        const uint32_t o = valid ? rl_owner_dev(recs[a].ns_id, world) : 0;
        const unsigned vmask = __ballot_sync(0xffffffffu, valid);
        if (valid) {
            const unsigned m = __match_any_sync(vmask, o);
            if (lane == (uint32_t)(__ffs(m) - 1)) wcnt[warp][o] += __popc(m);
        }
        __syncwarp();
    }
    __syncthreads();
    if (!SCATTER) {
        if (tid < world) {
            uint32_t tot = 0;
            for (int w = 0; w < RL_PART_WARPS; w++) tot += wcnt[w][tid];
            tile_cnt[blockIdx.x * 32 + tid] = tot;
        }
        return;
    }
    if (tid < world) {
        uint32_t run = owner_base[tid] + tile_cnt[blockIdx.x * 32 + tid];
        for (int w = 0; w < RL_PART_WARPS; w++) {
            const uint32_t c = wcnt[w][tid];
            wcnt[w][tid] = run;
            run += c;
        }
    }
    __syncthreads();
    for (uint32_t b = s0; b < s1; b += 32) {
        const uint32_t a = b + lane;
        const bool valid = a < s1;
        rl_record rec;
        uint32_t o = 0;
        if (valid) {
            rec = recs[a];
            o = rl_owner_dev(rec.ns_id, world);
        }
        const unsigned vmask = __ballot_sync(0xffffffffu, valid);
        if (valid) {
            const unsigned m = __match_any_sync(vmask, o);
            const int leader = __ffs(m) - 1;
            uint32_t basepos = 0;
            if ((int)lane == leader) {
                basepos = wcnt[warp][o];
                wcnt[warp][o] = basepos + __popc(m);
            }
            basepos = __shfl_sync(m, basepos, leader);
            const uint32_t pos = basepos + __popc(m & ((1u << lane) - 1));
            if (slot_cap == 0) {
                out_recs[pos] = rec;
                out_src[pos] = a;
            } else if (pos - o * slot_cap < slot_cap) {
                out_recs[pos] = rec;
                out_pos[a] = pos;
            } else {
                out_pos[a] = 0xFFFFFFFFu;  // block overflow (flagged by k_bucket_scan)
            }
        }
        __syncwarp();
    }
}

// single CTA: tile_cnt[t][o] -> exclusive prefix over tiles; owner totals -> owner_base
__global__ void k_bucket_scan(uint32_t num_tiles, uint32_t world, uint32_t* tile_cnt, uint32_t* owner_base,
                              unsigned long long* counts_out, uint32_t slot_cap, uint32_t* overflow) {
    __shared__ uint32_t tot[32];
    const uint32_t o = threadIdx.x;
    if (o < 32) {
        uint32_t run = 0;
        if (o < world)
            for (uint32_t t = 0; t < num_tiles; t++) {
                const uint32_t c = tile_cnt[t * 32 + o];
                tile_cnt[t * 32 + o] = run;
                run += c;
            }
        tot[o] = run;
    }
    __syncthreads();
    if (o == 0) {
        uint32_t run = 0;
        for (uint32_t w = 0; w < world; w++) {
            owner_base[w] = slot_cap ? w * slot_cap : run;
            counts_out[w] = tot[w];
            run += tot[w];
            if (slot_cap && tot[w] > slot_cap && overflow) atomicOr(overflow, 1u);
        }
    }
}

__global__ void k_gather_u8(uint32_t n, const uint8_t* __restrict__ in, const uint32_t* __restrict__ pos,
                            uint8_t* out) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = (pos[i] != 0xFFFFFFFFu) ? in[pos[i]] : (uint8_t)RL_VERDICT_ERROR;  // block overflow: not decided
}

// The lane byte of rl_record (top byte of key_hi) is opaque to the engine: the pipelined exchange
// returns the verdicts of an earlier step in it, so a step costs ONE all-to-all instead of two.
__global__ void k_lane_put(uint32_t n_slots, rl_record* recs, const uint8_t* __restrict__ lane_in) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_slots) reinterpret_cast<uint8_t*>(recs + i)[RL_RECORD_LANE_BYTE] = lane_in[i];
}

__global__ void k_lane_gather(uint32_t n, const rl_record* __restrict__ recs, const uint32_t* __restrict__ pos,
                              uint8_t* out) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = (pos[i] != 0xFFFFFFFFu) ? reinterpret_cast<const uint8_t*>(recs + pos[i])[RL_RECORD_LANE_BYTE] : (uint8_t)RL_VERDICT_ERROR;
}

__global__ void k_unpermute_u8(uint32_t n, const uint8_t* __restrict__ in, const uint32_t* __restrict__ src,
                               uint8_t* out) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[src[i]] = in[i];
}

