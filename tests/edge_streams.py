"""Seeded request streams that sit on the u64, clock and limit edges of the decision arithmetic (test
infrastructure only).  helpers.py's generators draw small values (max_value <= 2^40, deltas <= 7, round clock
steps); these draw the values where an implementation that saturates instead of wrapping, uses `<` for the
inclusive expiry bound or forgets the `checked_sub` guard gives a different answer than the reference:

  max_value   {0, 1, 2^32-1, 2^32, 2^63-1, 2^63, 2^64-2, 2^64-1, 3, 20}
  window_us   {0, 1, 1 s, 1 h, 2^40}, several windows inside one row (a live cell next to an expired one)
  deltas      CSR u64 {0, 1, 2^32-1, 2^32, 2^63, 2^64-1} + the amount that lands exactly on max_value (and +1),
              records u32 {0, 1, 2^31, 2^32-1}, compact 1..255
  clocks      now in {expiry-1, expiry, expiry+1} of the live counters a request touches, non-monotone steps,
              stamps just below the 2^62 bound of include/rl_engine.h
  keys        key_hi {0, 1, 0xFFFFFFFF} x key_lo {0, 1, 2^64-1}: 9 keys per variable set, so runs are long

The generator reads the oracle's table between batches (`dump`) to anchor clocks and deltas on the live state;
`preseed` builds an update batch that parks chosen counters a few deltas below 2^64, so that the following
batches wrap inside runs.  All arrays use the engine's dtypes (LIMIT_DESC_DTYPE, COUNTER_DTYPE, RECORD_DTYPE)."""
from __future__ import annotations

import numpy as np

from limitador_b200.engine import COUNTER_DTYPE, LIMIT_DESC_DTYPE, RECORD_DTYPE

M64 = (1 << 64) - 1
S = 1_000_000
T0 = 1_700_000_000_000_000
T_TOP = (1 << 62) - (1 << 41)  # near the top of the clock range: now + 2^40 windows still fit below 2^62
T_MAX = (1 << 62) - 1

EDGE_MAX = [0, 1, (1 << 32) - 1, 1 << 32, (1 << 63) - 1, 1 << 63, M64 - 1, M64, 3, 20]
EDGE_WIN = [0, 1, S, 3600 * S, 1 << 40]
CSR_DELTAS = [0, 1, (1 << 32) - 1, 1 << 32, 1 << 63, M64]
REC_HITS = [0, 1, 1 << 31, (1 << 32) - 1]
KEY_HI = [0, 1, 0xFFFFFFFF]
KEY_LO = [0, 1, M64]

_SHAPES = {  # (varset, qualified) per limit, the row shapes of helpers.mixed_limits
    "q1": [(1, 1)],
    "q4": [(1, 1)] * 4,
    "q2v": [(1, 1), (1, 1), (2, 1)],
    "uq": [(0, 0), (1, 1)],
    "u": [(0, 0), (0, 0)],
    "q3u2": [(1, 1), (0, 0), (1, 1), (2, 1), (0, 0)],
}


def _pick(rng, seq):
    """One element of a list of Python ints (numpy's choice would squeeze values >= 2^63 into int64)."""
    return int(seq[int(rng.integers(0, len(seq)))])


def _windows(rng, k):
    """k windows for the limits of one row: consecutive entries of EDGE_WIN from a random start, so that a row of
    several limits always mixes short (0 / 1 us) and long windows."""
    s = int(rng.integers(0, len(EDGE_WIN)))
    return [EDGE_WIN[(s + j) % len(EDGE_WIN)] for j in range(k)]


def edge_mixed_limits(n_ns=12, seed=0):
    """helpers.mixed_limits' row shapes (single-row, several rows, unqualified + qualified) with edge values."""
    rng = np.random.default_rng(seed)
    descs, lid = [], 0
    shapes = list(_SHAPES)
    for ns in range(n_ns):
        plan = _SHAPES[shapes[ns % len(shapes)]]
        wins = _windows(rng, len(plan))
        for (varset, q), win in zip(plan, wins):
            descs.append((lid, ns, varset, q, _pick(rng, EDGE_MAX), win))
            lid += 1
    return np.array(descs, dtype=LIMIT_DESC_DTYPE)


def edge_single_row_limits(cells, n_ns=9, seed=0):
    """Every namespace maps to one row (the record fast path, the sharded step): 1..cells limits on one
    variable set, every fourth namespace unqualified; edge values."""
    rng = np.random.default_rng(seed)
    descs, lid = [], 0
    for ns in range(n_ns):
        k = int(rng.integers(1, cells + 1))
        q = 0 if ns % 4 == 3 else 1
        for win in _windows(rng, k):
            descs.append((lid, ns, 1 if q else 0, q, _pick(rng, EDGE_MAX), win))
            lid += 1
    return np.array(descs, dtype=LIMIT_DESC_DTYPE)


class EdgeGen:
    """Batches over `descs` drawn against a snapshot of the oracle's table (`dump()` of the checker, taken by the
    caller between batches).  Pass the current descs after a limit update so "lands on max" follows it."""

    def __init__(self, descs, seed, t0=T0):
        self.rng = np.random.default_rng(seed)
        self.set_limits(descs)
        self.t = t0

    def set_limits(self, descs):
        self.descs = np.array(descs, dtype=LIMIT_DESC_DTYPE)
        self.lim = {int(d["limit_id"]): d for d in self.descs}
        self.by_ns = {}
        for d in self.descs:
            self.by_ns.setdefault(int(d["ns_id"]), []).append(d)
        self.nss = sorted(self.by_ns)

    # -- clocks ---------------------------------------------------------------------------------
    def _step(self):
        r = self.rng.random()
        if r < 0.12:  # non-monotone
            self.t -= int(self.rng.choice([1, 1000, 2 * S]))
        else:
            self.t += int(self.rng.choice([0, 0, 1, 1000, S, 3 * S]))
        self.t = min(max(self.t, 1), T_MAX)
        return self.t

    def _now(self, state, ctrs):
        """A clock reading for a request touching `ctrs`: half the time right on a live expiry of one of them."""
        exps = [state[c][1] for c in ctrs if c in state and state[c][1] > 1]
        if exps and self.rng.random() < 0.5:
            e = int(self.rng.choice(exps)) + int(self.rng.choice([-1, 0, 0, 1]))
            return min(max(e, 1), T_MAX)
        return self._step()

    def _land(self, state, ctr, now):
        """The delta that makes value_at(now) + delta == max_value of `ctr` (mod 2^64)."""
        v, e = state.get(ctr, (0, 0))
        v = 0 if e <= now else v
        return (int(self.lim[ctr[0]]["max_value"]) - v) & M64

    @staticmethod
    def state_of(dump):
        return {(lid, lo, hi): (val, exp) for lid, lo, hi, val, exp in dump}

    def _key(self):
        return _pick(self.rng, KEY_LO), int(self.rng.choice(KEY_HI))

    def _counters_of(self, ns, subset=True):
        lims = self.by_ns[ns]
        pick = list(range(len(lims)))
        if subset and self.rng.random() < 0.4:
            k = int(self.rng.integers(1, len(lims) + 1))
            pick = sorted(self.rng.choice(len(lims), size=k, replace=False).tolist())
        if self.rng.random() < 0.3:
            self.rng.shuffle(pick)
        vkeys, out = {}, []
        for j in pick:
            d = lims[j]
            if d["qualified"]:
                vs = int(d["varset_id"])
                if vs not in vkeys:
                    vkeys[vs] = self._key()
                lo, hi = vkeys[vs]
            else:
                lo, hi = 0, 0
            out.append((int(d["limit_id"]), lo, hi))
        return out

    # -- batches --------------------------------------------------------------------------------
    def csr(self, n, dump, uniform=None, subset=True, deltas=CSR_DELTAS):
        """CSR batch (off, ctrs, delta, now).  uniform: every request carries that delta (long closed-form runs)."""
        state = self.state_of(dump)
        off, ctrs = [0], []
        delta = np.zeros(n, dtype=np.uint64)
        now = np.zeros(n, dtype=np.uint64)
        for i in range(n):
            cs = self._counters_of(int(self.rng.choice(self.nss)), subset)
            ctrs += [(lid, 0, lo, hi) for lid, lo, hi in cs]
            off.append(len(ctrs))
            t = self._now(state, cs)
            now[i] = t
            if uniform is not None:
                delta[i] = uniform
            else:
                r = self.rng.random()
                if r < 0.3:
                    land = self._land(state, cs[int(self.rng.integers(0, len(cs)))], t)
                    delta[i] = (land + int(self.rng.integers(0, 2))) & M64
                elif r < 0.5:
                    delta[i] = int(self.rng.choice([1, 2, 3]))
                else:
                    delta[i] = _pick(self.rng, deltas)
        return (np.array(off, dtype=np.uint32), np.array(ctrs, dtype=COUNTER_DTYPE), delta, now)

    def records(self, n, dump, uniform=None, hits=REC_HITS):
        """32-byte records; hits_addend from `hits` and the u32 amounts that land on max_value."""
        state = self.state_of(dump)
        r = np.zeros(n, dtype=RECORD_DTYPE)
        for i in range(n):
            ns = int(self.rng.choice(self.nss))
            lo, hi = self._key()
            cs = [(int(d["limit_id"]), lo, hi) if d["qualified"] else (int(d["limit_id"]), 0, 0) for d in self.by_ns[ns]]
            t = self._now(state, cs)
            if uniform is not None:
                h = uniform
            else:
                x = self.rng.random()
                h = int(self.rng.choice(hits))
                if x < 0.3:
                    land = self._land(state, cs[int(self.rng.integers(0, len(cs)))], t) + int(self.rng.integers(0, 2))
                    if land < 1 << 32:
                        h = land
                elif x < 0.5:
                    h = int(self.rng.choice([1, 2, 3]))
            r[i] = (ns, h, lo, hi, t)
        return r

    def batch_clock(self, dump):
        """One clock reading for a whole batch: on a live expiry (-1, 0, +1) when there is one, else a step."""
        exps = [e for (_, _, _, _, e) in dump if e > 1]
        if exps and self.rng.random() < 0.7:
            self.t = min(max(int(self.rng.choice(exps)) + int(self.rng.choice([-1, 0, 1])), 1), T_MAX)
            return self.t
        return self._step()

    def compact_batch(self, n, dump):
        """Records for the 16-byte form: key_hi 0xFFFFFFFF on half of them, hits 1..255, one clock reading for the
        whole batch anchored on a live expiry when there is one.  Returns (records, now)."""
        t = self.batch_clock(dump)
        r = np.zeros(n, dtype=RECORD_DTYPE)
        r["ns_id"] = self.rng.choice(self.nss, size=n)
        r["hits_addend"] = np.where(self.rng.random(n) < 0.5, self.rng.integers(1, 256, n), self.rng.choice([1, 254, 255], n))
        r["key_lo"] = self.rng.choice(np.array(KEY_LO, dtype=np.uint64), size=n)
        r["key_hi"] = np.where(self.rng.random(n) < 0.5, 0xFFFFFFFF, self.rng.choice(KEY_HI, n)).astype(np.uint64)
        r["now_us"] = t
        return r, t

    def preseed(self, dump, gap=(1, 2, 3), per_ns=4, ds=(1, 3, 1 << 32, (1 << 32) - 1)):
        """A CSR update batch that parks counters of every namespace `k * d` below 2^64 (k in gap, d drawn from ds:
        the delta of the run that follows), so that the next batches wrap inside a run.  Returns (batch, d)."""
        state = self.state_of(dump)
        d = _pick(self.rng, ds)
        off, ctrs, delta, now = [0], [], [], []
        for ns in self.nss:
            for _ in range(per_ns):
                cs = self._counters_of(ns, subset=False)
                t = self._step()
                # update_counters adds the same delta to every counter of the request: aim at the first one
                v, e = state.get(cs[0], (0, 0))
                v = 0 if e <= t else v
                target = (M64 + 1 - int(self.rng.choice(gap)) * d) & M64
                ctrs += [(lid, 0, lo, hi) for lid, lo, hi in cs]
                off.append(len(ctrs))
                delta.append((target - v) & M64)
                now.append(t)
        return (np.array(off, dtype=np.uint32), np.array(ctrs, dtype=COUNTER_DTYPE),
                np.array(delta, dtype=np.uint64), np.array(now, dtype=np.uint64)), d

    def limit_updates(self, k=3):
        """New max_values for k live limits: below live values, 2^64-1 and 0.  Returns the changed descs."""
        idx = self.rng.choice(len(self.descs), size=min(k, len(self.descs)), replace=False)
        out = self.descs[idx].copy()
        for j in range(len(out)):
            out[j]["max_value"] = [2, M64, 0][j % 3]
        return out
