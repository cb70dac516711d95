// rl_core.h — data layout + per-row fixed-window semantics shared by every kernel.
//
// Everything here is `__host__ __device__` so the SAME functions that run inside the
// sm_100a kernels can be exercised by tests/emu (a sequential host driver used only by
// the CPU test-suite to check the batching algorithm; it is not part of the product
// library and the product never falls back to it).
//
// Reference semantics restated (paths relative to /root/reference/):
//   limitador/src/storage/atomic_expiring_value.rs:19-24,36-42,68-79,87-99
//   limitador/src/storage/in_memory.rs:20-35 (is_within_limits), :47-69 (update_counter),
//   :72-156 (check_and_update)
#pragma once
#include <stdint.h>

#ifdef __CUDACC__
#define RL_HD __host__ __device__ __forceinline__
#else
#define RL_HD inline
#endif

#define RL_NONE_U32 0xFFFFFFFFu
#define RL_MAX_CELLS 7          // cells per row: 16-B header + 7 x 16-B cells = 128 B
#define RL_MAX_CTRS_PER_REQ 16  // positions are packed in nibbles
#define RL_TOMB_HI 0xFFFFFFFFFFFFFFFFull

// device error codes (sticky max in RlBatchCtl::err)
enum : uint32_t {
    RL_DEV_OK = 0,
    RL_DEV_TABLE_FULL = 1,         // -> RL_TRANSIENT
    RL_DEV_UNKNOWN_LIMIT = 2,      // -> RL_FATAL (reference panics, in_memory.rs:107)
    RL_DEV_KEY_RANGE = 3,          // key_hi >= 2^32
    RL_DEV_TOO_MANY_COUNTERS = 4,  // > RL_MAX_CTRS_PER_REQ counters in one request
    RL_DEV_GROUP_SPLIT = 5,        // one request touches > RL_MAX_CELLS cells of one row (cannot happen)
    RL_DEV_EXCHANGE = 6,           // peer exchange: a rank's step flag did not arrive in time / a block fill is out of range
    RL_DEV_CLOCK = 7,              // now_us == 0: an entry stored at expiry 0 would read as absent (RlRow)
};

// Per-(row group, cell) limit parameters.  max_value lives here and never in the row,
// so update_limit (storage/mod.rs:67-83) can change it under live counters.
struct RlCellDesc {
    uint64_t max_value;
    uint64_t window_us;  // seconds * 1e6 (counter.rs:76-78)
    uint32_t limit_id;   // RL_NONE_U32 = undefined cell
    uint32_t qualified;  // 1 = limit has variables (counter.rs:108-110)
};

// Per-limit lookup (indexed by the caller's dense limit_id).
struct RlLimitDev {
    uint32_t group;  // 0 = undefined limit
    uint32_t cell;
    uint32_t ns_id;
    uint32_t qualified;
};

// Per-namespace lookup for the 32-B record format (limit set implied by ns_id).
struct RlNsDev {
    uint32_t mode;     // 0 = no limits (always allowed), 1 = single row, 2 = several rows
    uint32_t group;    // mode 1: the row group
    uint32_t cells;    // mode 1: packed cell list (see rl_pack_cells)
    uint32_t lim_off;  // offset into ns_limit_ids (registration order), mode 1 and 2
    uint32_t lim_cnt;
    uint32_t qualified_row;  // mode 1: 1 if the row is keyed by the request key, 0 if key = 0
    uint32_t _pad[2];
};

// One access = one request touching one row.  32 bytes.
//   hdr_hi = (group << 32) | key_hi32 ; hdr_hi == 0 marks an unused access slot
//   cells  = nibble k (k < n) is the k-th touched cell index; bits 28..30 = n; bit 31 = the
//            request has other accesses too (multi-row request)
//   posorig= nibble k: position of that cell in the request's processing order
//            (unqualified first, in_memory.rs:105,121); nibble 8+k... see helpers below
struct RlAccess {
    uint64_t key_lo;
    uint64_t hdr_hi;
    uint32_t req;
    uint32_t cells;
    uint64_t posorig;  // low 32 bits: 7 position nibbles; high 32 bits: 7 original-index nibbles
};

RL_HD uint32_t rl_cells_n(uint32_t cells) { return (cells >> 28) & 7u; }
RL_HD bool rl_cells_multi(uint32_t cells) { return (cells >> 31) != 0; }
RL_HD uint32_t rl_cells_at(uint32_t cells, uint32_t k) { return (cells >> (4 * k)) & 0xFu; }
RL_HD uint32_t rl_pos_at(uint64_t posorig, uint32_t k) { return (uint32_t)(posorig >> (4 * k)) & 0xFu; }
RL_HD uint32_t rl_orig_at(uint64_t posorig, uint32_t k) { return (uint32_t)(posorig >> (32 + 4 * k)) & 0xFu; }

// 64-bit mixer (splitmix64 / murmur3 finaliser constants).
RL_HD uint64_t rl_mix64(uint64_t x) {
    x ^= x >> 33;
    x *= 0xff51afd7ed558ccdULL;
    x ^= x >> 33;
    x *= 0xc4ceb9fe1a85ec53ULL;
    x ^= x >> 33;
    return x;
}
// Hash of the row identity (group, 96-bit key).  High bits pick the region, low bits the
// home row inside the region; the whole word is the in-CTA grouping tag.
RL_HD uint64_t rl_row_hash(uint64_t key_lo, uint64_t hdr_hi) {
    return rl_mix64(key_lo ^ rl_mix64(hdr_hi ^ 0x9e3779b97f4a7c15ULL));
}

// ---------------------------------------------------------------------------------------
// Row state held by the walker while it replays a key's requests in stream order.
// A QUALIFIED cell with expiry == 0 is logically absent ("the reference has no entry");
// now_us >= 1 is required so a live entry never has expiry 0.
template <int CELLS>
struct RlRow {
    uint64_t value[CELLS];
    uint64_t expiry[CELLS];
};

// value_at (atomic_expiring_value.rs:19-24,76-79): inclusive expiry bound.
RL_HD uint64_t rl_value_at(uint64_t value, uint64_t expiry, uint64_t now) {
    return (expiry <= now) ? 0 : value;
}
// ttl (atomic_expiring_value.rs:68-74)
RL_HD uint64_t rl_ttl(uint64_t expiry, uint64_t now) { return expiry > now ? expiry - now : 0; }

// update (atomic_expiring_value.rs:36-42 + :87-99). An absent qualified cell (expiry 0) is
// first created as (0, now+W) by the callers of update (in_memory.rs:50-57,122-127) and
// then updated, which yields (delta, now+W) — the same as the expired branch below.
template <int CELLS>
RL_HD void rl_cell_update(RlRow<CELLS>& row, uint32_t c, uint64_t delta, uint64_t window_us,
                          uint64_t now) {
    if (row.expiry[c] <= now) {
        row.expiry[c] = now + window_us;
        row.value[c] = delta;
    } else {
        row.value[c] += delta;
    }
}

// check_and_update for a request whose counters all live in THIS row
// (in_memory.rs:72-156).  Returns the processing-order position of the first limited
// counter, or RL_NONE_U32 (= Authorization::Ok, all counters incremented).
//   desc        : RlCellDesc[RL_MAX_CELLS+1] of the row group
//   rem/ttl     : per-request output base (indexed by original counter index), nullable
template <int CELLS>
RL_HD uint32_t rl_walk_check_single(RlRow<CELLS>& row, uint32_t& dirty, const RlCellDesc* desc,
                                    uint32_t cells, uint64_t posorig, uint64_t delta, uint64_t now,
                                    bool load_counters, uint64_t* rem, uint64_t* ttl) {
    const uint32_t n = rl_cells_n(cells);
    uint32_t first = RL_NONE_U32;
    for (uint32_t k = 0; k < n; k++) {
        const uint32_t c = rl_cells_at(cells, k);
        const RlCellDesc d = desc[c];
        if (d.qualified && row.expiry[c] == 0) {  // get_with_by_ref: insert (0, now+W), :122-127
            row.value[c] = 0;
            row.expiry[c] = now + d.window_us;
            dirty |= 1u << c;
        }
        const uint64_t v = rl_value_at(row.value[c], row.expiry[c], now);
        const uint64_t sum = v + delta;  // wraps like a release build
        const bool over = sum > d.max_value;
        if (load_counters) {
            const uint32_t oi = rl_orig_at(posorig, k);
            if (rem) rem[oi] = over ? 0 : d.max_value - sum;  // checked_sub, :88-89
            if (ttl) ttl[oi] = rl_ttl(row.expiry[c], now);    // pre-update ttl, :114-116,:134-136
        }
        if (over && first == RL_NONE_U32) {
            first = rl_pos_at(posorig, k);
            if (!load_counters) return first;  // early return, :110-112,:130-132
        }
    }
    if (first != RL_NONE_U32) return first;  // :141-143 — nothing incremented
    for (uint32_t k = 0; k < n; k++) {       // :146-153
        const uint32_t c = rl_cells_at(cells, k);
        rl_cell_update(row, c, delta, desc[c].window_us, now);
        dirty |= 1u << c;
    }
    return RL_NONE_U32;
}

// One access of a MULTI-row request.  `fl_in` is the request-level first-limited position
// assumed for this round (fixed-point iteration, DESIGN.md §"coupled requests"); the
// function returns the first limited position among THIS access's cells given the row's
// current state, and applies the side effects that follow from fl_in:
//   * !load_counters: counters at positions <= fl_in are looked up (created if absent);
//     later ones are never reached (early return).
//   * fl_in == NONE: every counter is incremented.
template <int CELLS>
RL_HD uint32_t rl_walk_check_multi(RlRow<CELLS>& row, uint32_t& dirty, const RlCellDesc* desc,
                                   uint32_t cells, uint64_t posorig, uint64_t delta, uint64_t now,
                                   bool load_counters, uint32_t fl_in, uint64_t* rem, uint64_t* ttl) {
    const uint32_t n = rl_cells_n(cells);
    uint32_t local_first = RL_NONE_U32;
    for (uint32_t k = 0; k < n; k++) {
        const uint32_t c = rl_cells_at(cells, k);
        const RlCellDesc d = desc[c];
        const uint32_t pos = rl_pos_at(posorig, k);
        const bool reached = load_counters || fl_in == RL_NONE_U32 || pos <= fl_in;
        if (reached && d.qualified && row.expiry[c] == 0) {
            row.value[c] = 0;
            row.expiry[c] = now + d.window_us;
            dirty |= 1u << c;
        }
        // an absent cell reads as 0 whether or not it was just created
        const uint64_t v = rl_value_at(row.value[c], row.expiry[c], now);
        const uint64_t sum = v + delta;
        const bool over = sum > d.max_value;
        if (load_counters) {
            const uint32_t oi = rl_orig_at(posorig, k);
            if (rem) rem[oi] = over ? 0 : d.max_value - sum;
            if (ttl) ttl[oi] = rl_ttl(row.expiry[c], now);
        }
        if (over && local_first == RL_NONE_U32) local_first = pos;
    }
    if (fl_in == RL_NONE_U32) {
        for (uint32_t k = 0; k < n; k++) {
            const uint32_t c = rl_cells_at(cells, k);
            rl_cell_update(row, c, delta, desc[c].window_us, now);
            dirty |= 1u << c;
        }
    }
    return local_first;
}

// update_counters (lib.rs:411-423 → in_memory.rs:47-69): unconditional.
template <int CELLS>
RL_HD void rl_walk_update(RlRow<CELLS>& row, uint32_t& dirty, const RlCellDesc* desc,
                          uint32_t cells, uint64_t delta, uint64_t now) {
    const uint32_t n = rl_cells_n(cells);
    for (uint32_t k = 0; k < n; k++) {
        const uint32_t c = rl_cells_at(cells, k);
        rl_cell_update(row, c, delta, desc[c].window_us, now);
        dirty |= 1u << c;
    }
}

// ---------------------------------------------------------------------------------------
// Run-length replay (DESIGN.md §3.3).  A key's requests are replayed in stream order, but
// not one at a time: starting at position `pos` of the key's request list with row state S,
//   * hypothesis A — "request i is denied under S and changes nothing": the longest prefix
//     of such requests is final as-is (a denied check leaves the state untouched,
//     in_memory.rs:141-143), whatever their deltas and timestamps;
//   * hypothesis B — "every request from pos up to and including i is allowed and none needs
//     a window reset or an insert": then request i sees S with the deltas of pos..i-1 added,
//     so the longest prefix for which that holds is final too (values only accumulate,
//     atomic_expiring_value.rs:41);
//   * otherwise request pos is applied alone with the sequential rule.
// Every step is exact, so the replay equals one-at-a-time execution; saturated hot keys
// (all denied) and hot keys far from their limit (all allowed) finish in one step.
template <int CELLS>
RL_HD bool rl_eval_deny_noeffect(const RlRow<CELLS>& S, const RlCellDesc* desc, uint32_t cells, uint64_t posorig,
                                 uint64_t delta, uint64_t now, bool load_counters) {
    RlRow<CELLS> tmp = S;
    uint32_t dirty = 0;
    const uint32_t fl =
        rl_walk_check_single<CELLS>(tmp, dirty, desc, cells, posorig, delta, now, load_counters, nullptr, nullptr);
    return fl != RL_NONE_U32 && dirty == 0;
}

// dsum = sum of the deltas of the run INCLUDING this request (wraps like the reference's u64 add).
template <int CELLS>
RL_HD bool rl_eval_allow_run(const RlRow<CELLS>& S, const RlCellDesc* desc, uint32_t cells, uint64_t dsum,
                             uint64_t now) {
    const uint32_t n = rl_cells_n(cells);
    for (uint32_t k = 0; k < n; k++) {
        const uint32_t c = rl_cells_at(cells, k);
        if (S.expiry[c] <= now) return false;  // absent or expired: needs insert / reset
        if (S.value[c] + dsum > desc[c].max_value) return false;
    }
    return true;
}

// update_counters analogue of hypothesis B: no limit test, only "no reset / insert needed".
template <int CELLS>
RL_HD bool rl_eval_update_run(const RlRow<CELLS>& S, uint32_t cells, uint64_t now) {
    const uint32_t n = rl_cells_n(cells);
    for (uint32_t k = 0; k < n; k++)
        if (S.expiry[rl_cells_at(cells, k)] <= now) return false;
    return true;
}

// State seen by a member of an allowed run: S plus the run's earlier deltas on the touched cells.
template <int CELLS>
RL_HD void rl_advance_run(RlRow<CELLS>& S, uint32_t cells, uint64_t dprev) {
    const uint32_t n = rl_cells_n(cells);
    for (uint32_t k = 0; k < n; k++) S.value[rl_cells_at(cells, k)] += dprev;
}

// ---------------------------------------------------------------------------------------
// Resolve one request's counters into accesses (one per distinct row), in the reference's
// processing order: unqualified counters first, then qualified, each in the given order
// (in_memory.rs:105,121).  Writes at most m accesses to acc[0..m) (unused ones get
// hdr_hi = 0) and returns the number of accesses, or a negative RL_DEV_* code.
struct RlCtrIn {
    uint32_t limit_id;
    uint64_t key_lo, key_hi;
};

template <class GetCtr>
RL_HD int rl_resolve_request(uint32_t req, uint32_t m, GetCtr get, const RlLimitDev* limits,
                             uint32_t limits_cap, bool unqualified_first, RlAccess* acc) {
    if (m > RL_MAX_CTRS_PER_REQ) return -(int)RL_DEV_TOO_MANY_COUNTERS;
    uint32_t grp[RL_MAX_CTRS_PER_REQ], cel[RL_MAX_CTRS_PER_REQ];
    uint64_t klo[RL_MAX_CTRS_PER_REQ], khi[RL_MAX_CTRS_PER_REQ];
    uint8_t order[RL_MAX_CTRS_PER_REQ];
    uint32_t npos = 0;
    // pass 0: unqualified, pass 1: qualified (single pass in given order if !unqualified_first)
    for (int pass = 0; pass < 2; pass++) {
        for (uint32_t j = 0; j < m; j++) {
            const RlCtrIn c = get(j);
            if (c.limit_id >= limits_cap) return -(int)RL_DEV_UNKNOWN_LIMIT;
            const RlLimitDev l = limits[c.limit_id];
            if (l.group == 0) return -(int)RL_DEV_UNKNOWN_LIMIT;
            if (unqualified_first ? ((int)(l.qualified != 0) != pass) : (pass != 0)) continue;
            if (l.qualified && (c.key_hi >> 32) != 0) return -(int)RL_DEV_KEY_RANGE;
            grp[j] = l.group;
            cel[j] = l.cell;
            klo[j] = l.qualified ? c.key_lo : 0;
            khi[j] = l.qualified ? c.key_hi : 0;
            order[npos++] = (uint8_t)j;
        }
    }
    uint32_t used = 0;  // bitmask of counters already assigned to an access
    uint32_t nacc = 0;
    for (uint32_t p = 0; p < npos; p++) {
        const uint32_t j = order[p];
        if (used & (1u << j)) continue;
        RlAccess a;
        a.key_lo = klo[j];
        a.hdr_hi = ((uint64_t)grp[j] << 32) | khi[j];
        a.req = req;
        uint32_t cells = 0, cnt = 0;
        uint64_t posorig = 0;
        for (uint32_t q = p; q < npos; q++) {
            const uint32_t jj = order[q];
            if (used & (1u << jj)) continue;
            if (grp[jj] != grp[j] || klo[jj] != klo[j] || khi[jj] != khi[j]) continue;
            if (cnt >= RL_MAX_CELLS) return -(int)RL_DEV_GROUP_SPLIT;
            cells |= cel[jj] << (4 * cnt);
            posorig |= (uint64_t)q << (4 * cnt);
            posorig |= (uint64_t)jj << (32 + 4 * cnt);
            used |= 1u << jj;
            cnt++;
        }
        a.cells = cells | (cnt << 28);
        a.posorig = posorig;
        acc[nacc++] = a;
    }
    if (nacc > 1)
        for (uint32_t x = 0; x < nacc; x++) acc[x].cells |= 0x80000000u;
    for (uint32_t x = nacc; x < m; x++) {
        acc[x].key_lo = 0;
        acc[x].hdr_hi = 0;
        acc[x].req = req;
        acc[x].cells = 0;
        acc[x].posorig = 0;
    }
    return (int)nacc;
}
