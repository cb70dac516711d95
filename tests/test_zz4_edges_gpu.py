"""The sm_100a kernels at the u64, clock and limit-update edges (tests/edge_streams.py) against the CPU oracle
replaying the same stream in the same order: verdicts, the first limited limit, remaining/ttl, the full table.
The device code carries its own copies of the arithmetic (hypotheses A/B of the run replay, the closed-form
run sums, rl_apply_check_smem / _update_smem, rl_query_counter, k_scan's remaining), so these run the edge
values through each entry point and assert that the path a case names actually ran."""
import numpy as np
import pytest

from limitador_b200 import Engine, EngineError
from limitador_b200.engine import COUNTER_DTYPE, LIMIT_DESC_DTYPE, RECORD_DTYPE, pack_records16
from tests import edge_streams as ES
from tests import helpers as H

pytestmark = pytest.mark.gpu
S = ES.S
U32_RUN = (1, 3, (1 << 32) - 1)  # run deltas a u32 hits_addend can carry


def _engine(descs, cells, flags=0, regions=8, max_batch=1 << 15):
    e = Engine(capacity_rows=1 << 14, cells_per_row=cells, max_batch=max_batch, regions=regions, flags=flags)
    e.limits_set(descs)
    return e


def _tables_equal(e, o, descs):
    assert H.normalise_dump(e.dump(), descs) == H.normalise_dump(o.dump(), descs), "counter tables differ"


def _set_limits(e, o, gen, descs, upd):
    """rl_limits_set on existing limits (max_value below live values, 2^64-1, 0), the oracle at the same point."""
    e.limits_set(upd)
    for u in upd:
        o.limit_set(int(u["limit_id"]), int(u["ns_id"]), int(u["max_value"]), int(u["window_us"]), bool(u["qualified"]))
    descs = descs.copy()
    for u in upd:
        descs["max_value"][descs["limit_id"] == u["limit_id"]] = u["max_value"]
    gen.set_limits(descs)
    return descs


def _preseed(e, o, gen, ds=U32_RUN):
    pre, d = gen.preseed(o.dump(), ds=ds)
    e.update_batch(*pre)
    o.batch_csr(2, *pre)
    return d


def _check_records(e, o, recs, lc, stride, tag):
    got = e.check_and_update_records(recs, lc, stride=stride)
    want = o.batch_records(0, recs, lc, stride)
    assert got[0].tolist() == want[0].tolist(), f"verdicts, {tag}"
    assert got[1].tolist() == want[1].tolist(), f"first limited, {tag}"
    if lc:
        assert got[2].tolist() == want[2].tolist(), f"remaining, {tag}"
        assert got[3].tolist() == want[3].tolist(), f"ttl, {tag}"


# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("cells", [1, 3, 7])
@pytest.mark.parametrize("load_counters", [False, True])
def test_records_default_path(cells, load_counters, monkeypatch):
    """k_main's replay (rl_apply_check_smem, the A/B run hypotheses) on wrapping runs, expiry rollovers and a
    limit lowered below live values between host calls."""
    monkeypatch.setenv("RL_HOT", "0")
    descs = ES.edge_single_row_limits(cells, seed=cells)
    e, o = _engine(descs, cells), H.oracle_with_limits(descs)
    gen = ES.EdgeGen(descs, 10 * cells + load_counters, t0=ES.T_TOP if cells == 3 else ES.T0)
    d = _preseed(e, o, gen)
    _tables_equal(e, o, descs)
    for b in range(6):
        recs = gen.records(3000, o.dump(), uniform=[None, d, None, 1, d, None][b])
        _check_records(e, o, recs, load_counters, cells, f"batch {b}")
        _tables_equal(e, o, descs)
        if b == 2:
            descs = _set_limits(e, o, gen, descs, gen.limit_updates(3))
    assert e.stats()["kernel_launches"] > 0 and e.stats()["hot_rows"] == 0


def test_hot_rows_carry_the_edges(monkeypatch):
    """k_hot: the hot keys take wrapping and saturated runs and the now == expiry rollovers."""
    monkeypatch.setenv("RL_HOT", "1")
    descs = ES.edge_single_row_limits(3, n_ns=3, seed=40)
    e, o = _engine(descs, 3, regions=4), H.oracle_with_limits(descs)
    gen = ES.EdgeGen(descs, 41)
    rng = np.random.default_rng(42)
    seen_hot = 0
    for b in range(7):
        if b in (1, 4):
            d = _preseed(e, o, gen)
        recs = gen.records(12000, o.dump(), uniform=d if b in (2, 5) else None)
        hot = rng.random(len(recs)) < 0.8
        hot_lo = np.where(rng.random(len(recs)) < 0.5, np.uint64(ES.M64), np.uint64(0))
        recs["key_lo"] = np.where(hot, hot_lo, recs["key_lo"])
        recs["key_hi"] = np.where(hot, np.uint64(0xFFFFFFFF), recs["key_hi"])
        recs["ns_id"] = np.where(hot, rng.integers(0, 3, len(recs)), recs["ns_id"])
        _check_records(e, o, recs, bool(b & 1), 3, f"batch {b}")
        _tables_equal(e, o, descs)
        seen_hot = max(seen_hot, e.stats()["hot_rows"])
    assert seen_hot > 0


def test_chained_commit_carries_the_edges(monkeypatch):
    monkeypatch.setenv("RL_HEAVY_MULT", "1")
    monkeypatch.setenv("RL_CHUNK", "128")
    monkeypatch.setenv("RL_HOT", "0")
    for cells in (1, 3):
        descs = ES.edge_single_row_limits(cells, seed=60 + cells)
        e, o = _engine(descs, cells, flags=4, regions=4), H.oracle_with_limits(descs)  # RL_FLAG_KERNEL_STATS
        gen = ES.EdgeGen(descs, 61 + cells)
        d = _preseed(e, o, gen)
        for b in range(4):
            recs = gen.records(6000, o.dump(), uniform=d if b % 2 else None)
            _check_records(e, o, recs, bool(b & 1), cells, f"cells {cells} batch {b}")
            _tables_equal(e, o, descs)
        st = e.stats()
        assert st["chained_chunks"] > 0 and st["ordered_chunks"] > 0


@pytest.mark.parametrize("cells", [3, 7])
@pytest.mark.parametrize("load_counters", [False, True])
def test_csr_coupled_requests(cells, load_counters):
    """The general form: multi-row requests through the fixed point with wrapping values, u64 deltas up to
    2^64-1 and the amounts that land on max_value."""
    descs = ES.edge_mixed_limits(n_ns=12, seed=70 + cells)
    e, o = _engine(descs, cells), H.oracle_with_limits(descs)
    gen = ES.EdgeGen(descs, 71 + cells + 2 * load_counters, t0=ES.T_TOP if load_counters else ES.T0)
    d = _preseed(e, o, gen, ds=(1, 3, 1 << 32, (1 << 32) - 1))
    for b in range(5):
        batch = gen.csr(2000, o.dump(), uniform=[None, d, None, 1, d][b])
        got = e.check_and_update_batch(*batch, load_counters)
        want = o.batch_csr(0, *batch, load_counters)
        assert got[0].tolist() == want[0].tolist(), f"verdicts, batch {b}"
        assert got[1].tolist() == want[1].tolist(), f"first limited, batch {b}"
        if load_counters:
            assert got[2].tolist() == want[2].tolist(), f"remaining, batch {b}"
            assert got[3].tolist() == want[3].tolist(), f"ttl, batch {b}"
        _tables_equal(e, o, descs)
        if b == 2:
            descs = _set_limits(e, o, gen, descs, gen.limit_updates(3))
    assert e.stats()["fixed_point_rounds"] >= 1


def test_update_is_within_limits_and_get_counters():
    """update pushes values past 2^64 (CSR and records); is_within_limits reads them (rl_query_counter's
    `max >= v + delta` on the wrapped sum); get_counters' remaining when value > max and ttl at now == expiry."""
    descs = ES.edge_mixed_limits(n_ns=12, seed=80)
    e, o = _engine(descs, 3), H.oracle_with_limits(descs)
    gen = ES.EdgeGen(descs, 81)
    ids = descs["limit_id"]
    for b in range(4):
        pre, _ = gen.preseed(o.dump(), per_ns=2)
        e.update_batch(*pre)
        o.batch_csr(2, *pre)
        batch = gen.csr(1500, o.dump())
        e.update_batch(*batch)
        o.batch_csr(2, *batch)
        _tables_equal(e, o, descs)
        batch = gen.csr(1500, o.dump())
        lim, fl = e.is_within_limits_batch(*batch)
        wl, wf, _, _ = o.batch_csr(1, *batch)
        assert lim.tolist() == wl.tolist() and fl.tolist() == wf.tolist(), f"is_within_limits (CSR), batch {b}"
        recs = gen.records(1500, o.dump())
        e.update_records(recs)
        o.batch_records(2, recs)
        _tables_equal(e, o, descs)
        recs = gen.records(1500, o.dump())
        lim, fl = e.is_within_limits_records(recs)
        wl, wf, _, _ = o.batch_records(1, recs)
        assert lim.tolist() == wl.tolist() and fl.tolist() == wf.tolist(), f"is_within_limits (records), batch {b}"
        _tables_equal(e, o, descs)  # read-only
        exps = sorted({x[4] for x in o.dump() if x[4] > 1})
        for t in [exps[len(exps) // 2] + k for k in (-1, 0, 1)] + [int(batch[3].max())]:
            assert e.get_counters(ids, t) == o.get_counters(ids, t), f"get_counters at {t}, batch {b}"
        if b == 1:
            descs = _set_limits(e, o, gen, descs, gen.limit_updates(4))
    mx = {int(x["limit_id"]): int(x["max_value"]) for x in descs}
    assert any(v > mx[l] for l, _, _, v, _ in o.dump()), "no counter above its limit: remaining never wrapped"


def test_compact_records_host_device_async():
    """The 16-byte form with key_hi = 0xFFFFFFFF and hits up to 255, one clock per batch on a live expiry."""
    import torch
    descs = ES.edge_single_row_limits(3, seed=90)
    e, o = _engine(descs, 3, flags=2), H.oracle_with_limits(descs)
    gen = ES.EdgeGen(descs, 91)
    _preseed(e, o, gen, ds=(1, 255))
    for b in range(9):
        recs, t = gen.compact_batch(4000, o.dump())
        r16 = pack_records16(recs)
        want = o.batch_records(0, recs)
        mem = b % 3
        if mem == 0:
            lim, fl = e.check_and_update_compact(r16, t)
        else:
            pin = (lambda x: x.cuda()) if mem == 1 else (lambda x: x.pin_memory())
            d = pin(torch.from_numpy(r16.view(np.int64).reshape(-1, 2).copy()))
            out = pin(torch.zeros(len(r16), dtype=torch.uint8))
            first = pin(torch.zeros(len(r16), dtype=torch.int32))
            e.check_and_update_compact_ptr(len(r16), d.data_ptr(), t, out.data_ptr(), mem, first.data_ptr())
            e.fence()
            e.sync()
            lim, fl = out.cpu().numpy(), first.cpu().numpy().astype(np.uint32)
        assert np.array_equal(lim, want[0]) and np.array_equal(fl, want[1]), f"batch {b} mem {mem}"
        _tables_equal(e, o, descs)


@pytest.mark.parametrize("fence_before_update", [False, True])
def test_pipelined_device_calls_and_limit_updates(fence_before_update):
    """RL_FLAG_PIPELINE device calls across the clock edges, with rl_limits_set issued between them.  Without a
    fence first, the engine's own ordering (ensure_ready syncs the pipeline before it re-uploads the tables) is
    what keeps the earlier calls on the old max_value and the later ones on the new one."""
    import torch
    descs = ES.edge_single_row_limits(3, seed=100)
    e, o = _engine(descs, 3, flags=2), H.oracle_with_limits(descs)
    gen = ES.EdgeGen(descs, 101 + fence_before_update)
    d = _preseed(e, o, gen)
    outs = []
    for b in range(8):
        recs = gen.records(4000, o.dump(), uniform=d if b % 3 == 1 else None)
        want = o.batch_records(0, recs)
        d_recs = torch.from_numpy(recs.view(np.int64).reshape(-1, 4).copy()).cuda()
        lim = torch.full((len(recs),), 9, dtype=torch.uint8, device="cuda")
        first = torch.zeros(len(recs), dtype=torch.int32, device="cuda")
        e.check_and_update_records_ptr(len(recs), d_recs.data_ptr(), lim.data_ptr(), 1, out_first_ptr=first.data_ptr(),
                                       stride=3)
        outs.append((d_recs, lim, first, want))
        if b in (2, 5):
            if fence_before_update:
                e.fence()
            descs = _set_limits(e, o, gen, descs, gen.limit_updates(3))
    e.fence()
    e.sync()
    for b, (_, lim, first, want) in enumerate(outs):
        assert np.array_equal(lim.cpu().numpy(), want[0]), f"verdicts, call {b}"
        assert np.array_equal(first.cpu().numpy().astype(np.uint32), want[1]), f"first limited, call {b}"
    _tables_equal(e, o, descs)


def test_sharded_exchange_against_one_global_oracle():
    """rl_shard_* on one GPU (world 2, lag 1): per step all sends, then all decides, then all collects; the oracle
    applies the steps in (step, source rank, source index) order."""
    import torch
    from limitador_b200 import exchange
    from limitador_b200.engine import Shard
    world, lag, batch, cells = 2, 1, 2048, 3
    descs = ES.edge_single_row_limits(cells, n_ns=16, seed=110)
    engines = [_engine(descs, cells, flags=2, max_batch=world * batch) for _ in range(world)]
    shards = [Shard(engines[r], r, world, batch, lag) for r in range(world)]
    for s in shards:
        s.connect_ptrs([x.slab for x in shards])
    o = H.oracle_with_limits(descs)
    gen = ES.EdgeGen(descs, 111)
    pre, d = gen.preseed(o.dump(), ds=U32_RUN)
    o.batch_csr(2, *pre)
    for eng in engines:  # each rank keeps the counters of the namespaces it owns
        ns_of = {int(x["limit_id"]): int(x["ns_id"]) for x in descs}
        off, ctrs, delta, now = pre
        keep = [i for i in range(len(delta)) if exchange.owner_of(ns_of[int(ctrs[off[i]]["limit_id"])], world) == engines.index(eng)]
        sub_off = np.concatenate([[0], np.cumsum([off[i + 1] - off[i] for i in keep])]).astype(np.uint32)
        sub_ctrs = np.concatenate([ctrs[off[i]:off[i + 1]] for i in keep]) if keep else np.zeros(0, COUNTER_DTYPE)
        eng.update_batch(sub_off, sub_ctrs, delta[keep], now[keep])
    steps, wants = [], []
    for st in range(6):
        t = gen.batch_clock(o.dump())
        row = []
        for r in range(world):
            recs = gen.records(batch, o.dump(), uniform=d if st % 2 else None)
            recs["now_us"] = t  # one clock for all ranks of a step
            row.append(recs)
            wants.append(o.batch_records(0, recs)[0])
        steps.append(row)
    d_recs = [[torch.from_numpy(x.view(np.int64).reshape(-1, 4).copy()).cuda() for x in row] for row in steps]
    d_out = [[torch.full((batch,), 7, dtype=torch.uint8, device="cuda") for _ in row] for row in steps]
    torch.cuda.synchronize()
    for st in range(len(steps)):
        for r in range(world):
            shards[r].send(batch, d_recs[st][r].data_ptr(), d_out[st][r].data_ptr())
        for r in range(world):
            shards[r].decide()
        for r in range(world):
            shards[r].collect()
    for s in shards:
        s.flush()
    for eng in engines:
        eng.sync()
    torch.cuda.synchronize()
    for st in range(len(steps)):
        for r in range(world):
            got = d_out[st][r].cpu().numpy()
            assert np.array_equal(got, wants[st * world + r]), f"step {st} rank {r}"
    union = [row for eng in engines for row in eng.dump()]
    assert H.normalise_dump(union, descs) == H.normalise_dump(o.dump(), descs)
    for s in shards:
        s.close()


# ---------------------------------------------------------------------------------------------------------------
def test_now_zero_is_refused_in_every_form():
    """1 <= now_us (include/rl_engine.h): a window-0 counter stamped at now 0 would be stored with expiry 0, which
    the table reads as "absent" while the reference keeps an entry.  Record forms mark the request
    RL_VERDICT_ERROR and report the error; CSR forms refuse the call before the table is touched."""
    import torch
    descs = np.array([(0, 0, 1, 1, 5, 0), (1, 1, 0, 0, 5, 0), (2, 2, 1, 1, 5, 60 * S)], dtype=LIMIT_DESC_DTYPE)
    recs = np.zeros(48, dtype=RECORD_DTYPE)
    recs["ns_id"] = np.arange(48) % 3
    recs["hits_addend"] = 1
    recs["key_lo"] = 1 + np.arange(48) % 4
    recs["now_us"] = H.T0
    bad = recs.copy()
    bad["now_us"][[5, 30]] = 0
    good = np.ones(48, dtype=bool)
    good[[5, 30]] = False
    # 32-byte records, device memory: the two requests read RL_VERDICT_ERROR, the others are decided
    e, o = _engine(descs, 1, flags=2), H.oracle_with_limits(descs)
    dv = torch.from_numpy(bad.view(np.int64).reshape(-1, 4).copy()).cuda()
    out = torch.zeros(48, dtype=torch.uint8, device="cuda")
    e.check_and_update_records_ptr(48, dv.data_ptr(), out.data_ptr(), 1, stride=1)
    with pytest.raises(EngineError, match="now_us"):
        e.sync()
    got = out.cpu().numpy()
    assert got[5] == 0xFF and got[30] == 0xFF
    assert np.array_equal(got[good], o.batch_records(0, recs[good])[0])
    _tables_equal(e, o, descs)
    # 32-byte records, host memory: check_and_update and update report it
    for call in (lambda x: x.check_and_update_records(bad, False, stride=1), lambda x: x.update_records(bad)):
        with pytest.raises(EngineError, match="now_us"):
            call(_engine(descs, 1))
    # CSR forms, host and device memory: refused before the table is touched
    off = np.arange(4, dtype=np.uint32)
    ctrs = np.array([(0, 0, 7, 0), (1, 0, 0, 0), (2, 0, 7, 0)], dtype=COUNTER_DTYPE)
    delta = np.ones(3, dtype=np.uint64)
    now = np.array([H.T0, 0, H.T0], dtype=np.uint64)
    e2 = _engine(descs, 1)
    before = e2.dump()
    for call in (lambda: e2.check_and_update_batch(off, ctrs, delta, now, True), lambda: e2.update_batch(off, ctrs, delta, now),
                 lambda: e2.is_within_limits_batch(off, ctrs, delta, now)):
        with pytest.raises(EngineError, match="before the table was touched"):
            call()
        assert e2.dump() == before
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).copy()).cuda()
    d_off, d_ctrs, d_delta, d_now = t(off), t(ctrs), t(delta), t(now)
    d_lim = torch.zeros(3, dtype=torch.uint8, device="cuda")
    L = e2._lib
    for st in (L.rl_check_and_update_batch(e2._h, 3, d_off.data_ptr(), d_ctrs.data_ptr(), d_delta.data_ptr(), d_now.data_ptr(),
                                          0, 1, d_lim.data_ptr(), None, None, None),
               L.rl_update_batch(e2._h, 3, d_off.data_ptr(), d_ctrs.data_ptr(), d_delta.data_ptr(), d_now.data_ptr(), 1)):
        assert st != 0 and "before the table was touched" in L.rl_last_error(e2._h).decode()
        assert e2.dump() == before
    # the corrected batch goes through and matches the oracle
    now[1] = H.T0
    o2 = H.oracle_with_limits(descs)
    assert e2.check_and_update_batch(off, ctrs, delta, now)[0].tolist() == o2.batch_csr(0, off, ctrs, delta, now)[0].tolist()
    _tables_equal(e2, o2, descs)
