"""The decision arithmetic at its u64, clock and limit-update edges (tests/edge_streams.py), on the CPU:

  * the C oracle against the Python restatement of the reference (tests/spec_model.py), every mode;
  * the host emulator of the kernels' batching algorithm (tests/emu/emu.cpp over rl_core.h) against the oracle,
    cells 1/3/7, both load_counters values, coupled requests, limit updates under live counters;
  * a mutation check: single-line mutants of the shared arithmetic, built with g++, must all be told apart
    from the oracle by the edge streams.

Measured when the edge streams were added: helpers.random_csr_stream (the streams of test_emu_algorithm.py)
catches three of the five mutants (`sum >= max`, the unguarded `max - sum` for remaining, the allow-run test on
the request's delta instead of the run's sum) and misses two: `expiry < now` in rl_value_at and the saturating
add (no stream lands on an expiry or wraps a u64).  test_random_streams_miss_what_the_edge_streams_catch
keeps that measurement honest."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest

from tests import edge_streams as ES
from tests import helpers as H
from tests.test_oracle_vs_spec import both, spec_batch

ROOT = os.path.dirname(H.HERE)


def _limit_set(targets, d):
    for t in targets:
        t.limit_set(int(d["limit_id"]), int(d["ns_id"]), int(d["max_value"]), int(d["window_us"]), bool(d["qualified"]))


def _apply_limit_updates(descs, upd):
    descs = descs.copy()
    for u in upd:
        descs["max_value"][descs["limit_id"] == u["limit_id"]] = u["max_value"]
    return descs


# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("seed", range(6))
def test_oracle_equals_the_python_spec_on_edge_streams(seed):
    descs = ES.edge_mixed_limits(n_ns=int([6, 12][seed % 2]), seed=seed)
    o, s = both(descs)
    gen = ES.EdgeGen(descs, 50 + seed, t0=ES.T_TOP if seed % 3 == 2 else ES.T0)
    pre, d = gen.preseed(o.dump())
    o.batch_csr(2, *pre)
    spec_batch(s, 2, *pre, False)
    assert H.normalise_dump(o.dump(), descs) == H.normalise_dump(s.dump(), descs), "state after the preseed"
    plan = [(0, False, d), (0, True, None), (1, False, None), (2, False, None), (0, True, d), (0, False, None),
            (1, False, d), (0, True, 1), (2, False, d), (0, False, 1)]
    for b, (mode, lc, uni) in enumerate(plan):
        batch = gen.csr(300, o.dump(), uniform=uni)
        got = o.batch_csr(mode, *batch, lc)
        want = spec_batch(s, mode, *batch, lc)
        assert np.array_equal(got[0], want[0]), f"verdicts, batch {b} mode {mode}"
        if mode != 2:
            assert np.array_equal(got[1], want[1]), f"first limited, batch {b} mode {mode}"
        if lc:
            assert np.array_equal(got[2], want[2]), f"remaining, batch {b}"
            assert np.array_equal(got[3], want[3]), f"ttl, batch {b}"
        assert H.normalise_dump(o.dump(), descs) == H.normalise_dump(s.dump(), descs), f"state, batch {b}"
        t = int(batch[3].max())
        ids = [int(x) for x in descs["limit_id"]]
        for tt in (t, t + 1, int(batch[3][-1])):
            assert sorted(o.get_counters(ids, tt)) == s.get_counters(ids, tt), f"get_counters, batch {b}"
        if b in (3, 7):  # max_value moves under live counters: below them, to 2^64-1, to 0
            upd = gen.limit_updates(3)
            for u in upd:
                _limit_set((o, s), u)
            descs = _apply_limit_updates(descs, upd)
            gen.set_limits(descs)


def test_edge_streams_reach_the_edges():
    """The generator does what it is for: wrapped values, requests on an expiry, values above a lowered limit."""
    descs = ES.edge_mixed_limits(n_ns=12, seed=1)
    o = H.oracle_with_limits(descs)
    gen = ES.EdgeGen(descs, 7)
    pre, d = gen.preseed(o.dump())
    o.batch_csr(2, *pre)
    on_expiry = wrapped = extreme = 0
    for b in range(6):
        before = {(l, lo, hi): (v, e) for l, lo, hi, v, e in o.dump()}
        off, ctrs, delta, now = gen.csr(300, o.dump(), uniform=d if b % 2 else None)
        for i in range(len(delta)):
            for c in ctrs[off[i]:off[i + 1]]:
                k = (int(c["limit_id"]), int(c["key_lo"]), int(c["key_hi"]))
                if k in before and before[k][1] == int(now[i]):
                    on_expiry += 1
        extreme += sum(1 for x in delta.tolist() if x in (0, ES.M64))
        o.batch_csr(0, off, ctrs, delta, now)
        after = {(l, lo, hi): (v, e) for l, lo, hi, v, e in o.dump()}
        wrapped += sum(1 for k, (v, e) in after.items() if k in before and before[k][1] == e and v < before[k][0])
    assert on_expiry > 20 and wrapped > 0 and extreme > 0
    upd = gen.limit_updates(3)
    for u in upd:
        _limit_set((o,), u)
    mx = {int(x["limit_id"]): int(x["max_value"]) for x in _apply_limit_updates(descs, upd)}
    assert any(v > mx[l] for l, _, _, v, _ in o.dump())


# ---------------------------------------------------------------------------------------------------------------
def _drive(emu, orc, descs, cells, lc, seed, nb=10, n=250):
    """Emulator vs oracle over one edge run; returns None or the first difference."""
    gen = ES.EdgeGen(descs, seed, t0=ES.T_TOP if seed % 2 else ES.T0)
    pre, d = gen.preseed(orc.dump())
    emu.batch_csr(2, *pre)
    orc.batch_csr(2, *pre)
    rounds = 0
    for b in range(nb):
        mode = 2 if b % 5 == 4 else 0
        uni = [None, d, None, 1, d][b % 5]
        batch = gen.csr(n, orc.dump(), uniform=uni)
        e = emu.batch_csr(mode, *batch, lc)
        o = orc.batch_csr(mode, *batch, lc)
        rounds = max(rounds, emu.rounds)
        if mode == 0:
            if e[0].tolist() != o[0].tolist():
                return f"verdicts, batch {b}"
            if e[1].tolist() != o[1].tolist():
                return f"first-limited limit, batch {b}"
            if lc and (e[2].tolist() != o[2].tolist() or e[3].tolist() != o[3].tolist()):
                return f"remaining/ttl, batch {b}"
        if H.normalise_dump(emu.dump(), descs) != H.normalise_dump(orc.dump(), descs):
            return f"table, batch {b}"
        if b == nb // 2:  # limit updates under live counters, at the same position for both
            upd = gen.limit_updates(3)
            for u in upd:
                _limit_set((orc,), u)
            descs = _apply_limit_updates(descs, upd)
            gen.set_limits(descs)
            limits, desc, ngroups = H.assign_tables(descs, cells)
            emu.L.emu_set_tables(emu.h, H._p(limits), len(limits), H._p(desc), ngroups)
    emu.max_rounds = rounds
    return None


@pytest.mark.parametrize("cells", [1, 3, 7])
@pytest.mark.parametrize("load_counters", [False, True])
@pytest.mark.parametrize("seed", [0, 1])
def test_emulator_equals_oracle_on_edge_streams(cells, load_counters, seed):
    descs = ES.edge_mixed_limits(n_ns=12, seed=10 + seed)
    emu = H.Emu(descs, cells)
    err = _drive(emu, H.oracle_with_limits(descs), descs, cells, load_counters, 100 * cells + seed)
    assert err is None, err
    assert emu.max_rounds >= 1  # coupled requests ran the fixed point with wrapping values


# ---------------------------------------------------------------------------------------------------------------
# Single-line mutants of the shared arithmetic.  (file, original line, mutated line)
MUTANTS = {
    "value_at_lt": ("rl_core.h", "return (expiry <= now) ? 0 : value;", "return (expiry < now) ? 0 : value;"),
    "over_ge": ("rl_core.h", "const bool over = sum > d.max_value;", "const bool over = sum >= d.max_value;"),
    "saturating_add": ("rl_core.h", "const uint64_t sum = v + delta;  // wraps like a release build",
                       "const uint64_t sum = (v + delta < v) ? ~0ull : v + delta;"),
    "remaining_unguarded": ("rl_core.h", "if (rem) rem[oi] = over ? 0 : d.max_value - sum;",
                            "if (rem) rem[oi] = d.max_value - sum;"),
    # rl_eval_allow_run only sees the run's sum; the call site is where the per-request delta could slip in
    "allow_run_delta": ("emu.cpp", "rl_eval_allow_run<RL_MAX_CELLS>(st, desc, A.cells, P[i] - pbase, now[A.req]);",
                        "rl_eval_allow_run<RL_MAX_CELLS>(st, desc, A.cells, delta[A.req], now[A.req]);"),
}


def _load_emu(so):
    L = C.CDLL(so)
    vp = C.c_void_p
    L.emu_create.restype = vp
    L.emu_create.argtypes = [C.c_int]
    L.emu_set_tables.argtypes = [vp, vp, C.c_uint32, vp, C.c_uint32]
    L.emu_batch_csr.argtypes = [vp, C.c_int, C.c_uint32, vp, vp, vp, vp, C.c_int, vp, vp, vp, vp, vp]
    L.emu_dump.restype = C.c_uint64
    L.emu_dump.argtypes = [vp, C.c_uint64, vp, vp, vp, vp, vp]
    return L


class _MutantEmu(H.Emu):
    def __init__(self, L, descs, cells):
        self.L = L
        self.h = L.emu_create(cells)
        limits, desc, ngroups = H.assign_tables(descs, cells)
        L.emu_set_tables(self.h, H._p(limits), len(limits), H._p(desc), ngroups)
        self.rounds = 0

    def batch_csr(self, mode, off, ctrs, delta, now_us, load_counters=False):
        try:
            return super().batch_csr(mode, off, ctrs, delta, now_us, load_counters)
        except AssertionError:  # a mutant may fail to converge: that is a difference too
            n = len(delta)
            return np.full(n, 2, np.uint8), np.full(n, 0, np.uint32), np.zeros(len(ctrs), np.uint64), np.zeros(len(ctrs), np.uint64)


@pytest.fixture(scope="module")
def mutant_libs(tmp_path_factory):
    """g++ builds of emu.cpp, one per mutant, from copies that keep the tree's relative include layout."""
    base = tmp_path_factory.mktemp("mutants")
    src_core = os.path.join(ROOT, "limitador_b200", "csrc", "rl_core.h")
    src_emu = os.path.join(H.HERE, "emu", "emu.cpp")
    procs = {}
    for name, (fname, old, new) in MUTANTS.items():
        d = base / name
        os.makedirs(d / "tests" / "emu")
        os.makedirs(d / "limitador_b200" / "csrc")
        shutil.copy(src_core, d / "limitador_b200" / "csrc" / "rl_core.h")
        shutil.copy(src_emu, d / "tests" / "emu" / "emu.cpp")
        target = d / ("limitador_b200/csrc/rl_core.h" if fname == "rl_core.h" else "tests/emu/emu.cpp")
        text = target.read_text()
        assert text.count(old) >= 1, f"mutant {name}: line not found"
        target.write_text(text.replace(old, new, 1))
        so = str(d / "librl_emu.so")
        procs[name] = (so, subprocess.Popen(["g++", "-O1", "-std=c++17", "-fPIC", "-shared", "-o", so,
                                             str(d / "tests" / "emu" / "emu.cpp")]))
    out = {}
    for name, (so, p) in procs.items():
        assert p.wait() == 0, f"mutant {name} does not compile"
        out[name] = _load_emu(so)
    return out


def _edge_catches(L):
    for cells, lc, seed in [(3, True, 0), (1, False, 1), (7, True, 2), (3, False, 3)]:
        descs = ES.edge_mixed_limits(n_ns=12, seed=10 + seed)
        if _drive(_MutantEmu(L, descs, cells), H.oracle_with_limits(descs), descs, cells, lc, 100 * cells + seed):
            return True
    return False


def _random_catches(L):
    for cells, lc, seed in [(1, False, 0), (3, True, 1), (7, True, 2)]:  # test_emu_algorithm's streams
        descs = H.mixed_limits(n_ns=12, seed=seed)
        emu, orc = _MutantEmu(L, descs, cells), H.oracle_with_limits(descs)
        for b in range(6):
            batch = H.random_csr_stream(descs, 300, seed * 100 + b, n_keys=3, monotone=(b % 2 == 0))
            e, o = emu.batch_csr(0, *batch, lc), orc.batch_csr(0, *batch, lc)
            if any(x.tolist() != y.tolist() for x, y in zip(e, o) if lc or x.dtype != np.uint64) or \
                    H.normalise_dump(emu.dump(), descs) != H.normalise_dump(orc.dump(), descs):
                return True
    return False


def test_edge_streams_catch_every_mutant(mutant_libs):
    missed = [name for name, L in mutant_libs.items() if not _edge_catches(L)]
    assert missed == [], f"mutants the edge streams do not tell apart from the oracle: {missed}"


def test_random_streams_miss_what_the_edge_streams_catch(mutant_libs):
    """The gap the edge streams close, as measured (module docstring): the older random streams miss two mutants."""
    missed = sorted(name for name, L in mutant_libs.items() if not _random_catches(L))
    assert missed == ["saturating_add", "value_at_lt"]
