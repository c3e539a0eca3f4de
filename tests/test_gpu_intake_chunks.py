"""The pipelined column intake (pqb_suite_run_columns / pqb_suite_run_record_batch) on a panel of several transfer chunks.

Host threads copy the caller's columns into pinned staging while the GPU works: chunk c goes to the device once every
column of its symbols is staged, and its null bookkeeping (starts, flags, validity words, block lists) is prepared for
that chunk alone.  2,536 x 5,040 (the benchmark's row length) is four chunks of 832, 832, 832 and 40 symbols, 80 symbol
blocks with an 8-symbol block 79 in the last chunk.  Every run is compared bit for bit, values and validity, with the
ungated whole-panel path (set_column + run_host) and the device path (compute: whole-panel preparation, symbol
compaction), and the chunk-edge and flagged symbols with the oracle's null rules."""
import ctypes as C

import numpy as np
import pyarrow as pa
import pytest

import synth
import tolerances as T
from oracle import pqo
from test_gpu_nulls import _check_symbol_against_the_oracle
from test_gpu_nulls_groups import DEFAULTS, expected, _outputs_of

pytestmark = pytest.mark.gpu

F = ("close", "high", "low", "volume")
S, NB = 2536, 5040
PITCH = -(-NB // 16) * 16
CS = max(32, (32 << 20) // (PITCH * 8) // 32 * 32)          # symbols per transfer chunk (engine.cu, pqb_panel_create)
N_CHUNKS = -(-S // CS)
SAMPLES = (0, 831, 832, 1663, 1664, 2495, 2496, 2535)      # the first and last symbol of every chunk
BLOCK = 32


@pytest.fixture(scope="module")
def pq():
    import polars_quant_b200 as pq
    return pq


@pytest.fixture(scope="module")
def N():
    from polars_quant_b200 import _native as N
    return N


@pytest.fixture(scope="module")
def d():
    return synth.ohlcv(S, NB, seed=0x1A7E)


def _nulls(chunks=(0, 1, 2, 3), variant=0):
    """Halts, delistings and late fields in the listed chunks only (validity per field, [S, NB] bool)."""
    ok = {f: np.ones((S, NB), bool) for f in F}

    def every(s, cols):
        for f in F:
            ok[f][s, cols] = False
    if 0 in chunks:
        ok["close"][831, 2000:2010] = False                 # a halt in the last symbol of chunk 0
        every(5, slice(0, 300))                             # listed later: a start, block 0 stays plain
    if 1 in chunks:
        if variant == 0:
            every(832, slice(4500, None))                   # delisted, first symbol of chunk 1; the rest of it clean
        else:
            every(1100, slice(1000, 1003))
            ok["volume"][1663, :77] = False                 # volume listed later than the prices, last symbol of chunk 1
    if 2 in chunks:
        for j in range(26):                                 # one symbol in each of blocks 52..77: every block of chunk 2
            s, t = 1664 + BLOCK * j + (7 * j) % BLOCK, 200 + 180 * j
            if j % 4 == 0:
                ok["close"][s, t] = False
            elif j % 4 == 1:
                every(s, slice(t, t + 5))
            elif j % 4 == 2:
                every(s, slice(t, None))
            else:
                ok["volume"][s, :t] = False
    if 3 in chunks:
        every(2500, slice(0, 600))                          # block 78: listed later only, stays plain
        ok["high"][2533, :40] = False                       # block 79 (8 symbols): high starts later, low halts
        ok["low"][2533, 3000] = False
    return ok


def _null_rows(ok):
    return sorted(set(np.nonzero(~np.logical_and.reduce([ok[f].all(axis=1) for f in F]))[0].tolist()))


def _flagged_blocks(ok):
    """Symbol blocks the engine sends through the null-aware kernel: a null after a field's first valid bar, or fields
    of one symbol that start on different bars."""
    out = set()
    for s in _null_rows(ok):
        first = [int(np.argmax(ok[f][s])) if ok[f][s].any() else NB for f in F]
        if len(set(first)) > 1 or any(not ok[f][s][a:].all() for f, a in zip(F, first)):
            out.add(s // BLOCK)
    return out


def _refs(pq, d, ok):
    """pqb_col_ref records of every (symbol, field), values in d's own rows, a validity bitmap only for rows with nulls."""
    rec, keep = pq.Panel.field_refs(d["close"], d["high"], d["low"], d["volume"])
    for i, f in enumerate(F):
        bad = np.nonzero(~ok[f].all(axis=1))[0]
        if len(bad):
            bits = np.packbits(ok[f][bad], axis=1, bitorder="little")
            keep.append(bits)
            rec["validity"][i * S + bad] = np.uint64(bits.ctypes.data) + np.arange(len(bad), dtype=np.uint64) * np.uint64(bits.strides[0])
    return rec, keep


def _staged(pq, d, ok, outputs_mask):
    """A panel given the columns one by one (pqb_panel_set_column)."""
    p = pq.Panel(S, NB, outputs_mask=outputs_mask)
    for s in range(S):
        for f in F:
            p.set_column(s, f, d[f][s], validity=None if ok[f][s].all() else np.packbits(ok[f][s], bitorder="little"))
    return p


def _same(N, a, b, mask, what):
    """Result planes of panels a and b: identical validity, identical bits (any NaN equals any NaN)."""
    for k, name in enumerate(N.OUTPUT_NAMES):
        if not mask >> k & 1:
            continue
        va, vb = a.host_output(k), b.host_output(k)
        if not np.array_equal(va.view(np.uint64), vb.view(np.uint64)):
            bad = ~T.same_bits(va, vb)
            assert not bad.any(), f"{what}: {name} values differ at {np.argwhere(bad)[:5].tolist()}"
        ka, kb = a.host_validity(k), b.host_validity(k)
        assert np.array_equal(ka, kb), f"{what}: {name} validity differs at {np.argwhere(ka != kb)[:5].tolist()}"


class Reference:
    """The ungated whole-panel path (set_column + run_host) of the given columns, checked once against compute()."""

    def __init__(self, pq, N, d, ok, params, mask):
        self.panel = _staged(pq, d, ok, mask)
        self.panel.run_host(params)
        dev = _staged(pq, d, ok, mask)
        dev.compute(params)
        _same(N, self.panel, dev, mask, "run_host vs compute")
        dev.close()

    def close(self):
        self.panel.close()


def _oracle_rows(res, d, ok, rows):
    """The 21 suite outputs of the given symbols against the oracle: a symbol whose fields share one first valid bar and
    have no later null is the oracle's dense computation from that bar, any other one follows the reference's null rules."""
    for s in rows:
        first = [int(np.argmax(ok[f][s])) for f in F]
        if len(set(first)) == 1 and all(ok[f][s][first[0]:].all() for f in F):
            a = first[0]
            out, okk, _ = pqo.suite_panel(*(d[f][s:s + 1, a:] for f in F))
            for j, name in enumerate(pqo.OUTPUT_NAMES):
                fv, fk = np.full(NB, np.nan), np.zeros(NB, bool)
                fv[a:], fk[a:] = out[j, 0], okk[j, 0]
                nbad, msg = T.compare(name, res[name][0][s], res[name][1][s], fv, fk)
                assert nbad == 0, f"symbol {s}: {msg}"
        else:
            _check_symbol_against_the_oracle(res, s, d, ok, NB)


def test_clean_panel_over_four_chunks_on_every_thread_count(pq, N, d):
    assert (CS, N_CHUNKS, S - (N_CHUNKS - 1) * CS) == (832, 4, 40)
    mask = (1 << N.N_SUITE_OUTPUTS) - 1
    ok = _nulls(chunks=())
    ref = Reference(pq, N, d, ok, N.default_params(), mask)
    refs, keep = _refs(pq, d, ok)
    p = pq.Panel(S, NB)
    nb, _ = p.tiled_shape()
    assert nb == 80
    for threads in (1, 2, 6, 0):
        p.run_columns(refs, threads=threads)
        assert p.last_launches() >= 3 * N_CHUNKS            # a pack, a suite launch and an unpack per chunk at least
        _same(N, p, ref.panel, mask, f"run_columns threads={threads}")
    _oracle_rows(p.outputs(), d, ok, SAMPLES)
    p.close(); ref.close()


KERNELS = {
    "full": lambda N: (N.default_params(), (1 << N.N_SUITE_OUTPUTS) - 1),
    "base": lambda N: (N.default_params(indicators=N.IND["ema"] | N.IND["kdj"] | N.IND["atr"]),
                       sum(1 << N.OUTPUT_NAMES.index(n) for n in ("ema", "atr", "kdj_k", "kdj_d", "kdj_j"))),
    "extras": lambda N: (N.default_params(indicators=N.IND_ALL | N.IND_EXTRA["dm"] | N.IND_EXTRA["aroon"] | N.IND_EXTRA["mom"], **DEFAULTS),
                         sum(1 << N.OUTPUT_NAMES.index(n) for n in N.OUTPUT_NAMES[:N.N_SUITE_OUTPUTS] + ["mom", "aroon_up", "aroon_down"]
                             + list(_outputs_of("dm")))),
}


@pytest.mark.parametrize("kernel", list(KERNELS))
def test_nulls_arriving_chunk_by_chunk(pq, N, d, kernel):
    """Nulls in the last symbol of chunk 0, the first symbol of chunk 1 (the rest of it clean: plain and null-aware launches
    side by side), one symbol in every block of chunk 2 (the null-aware launch alone) and in the 8-symbol block 79 (block 78
    clean).  The full suite runs the specialised null-aware kernel, EMA + KDJ + ATR the general one, the suite + DM, AROON
    and MOM two launches per block kind."""
    params, mask = KERNELS[kernel](N)
    ok = _nulls()
    flagged = _flagged_blocks(ok)
    assert {25, 26, 79} <= flagged and set(range(52, 78)) <= flagged and not {0, 27, 51, 78} & flagged
    ref = Reference(pq, N, d, ok, params, mask)
    refs, keep = _refs(pq, d, ok)
    p = pq.Panel(S, NB, outputs_mask=mask)
    p.run_columns(refs, params, threads=2)
    assert p.last_launches() >= 3 * N_CHUNKS
    _same(N, p, ref.panel, mask, f"{kernel}: run_columns")
    rows = sorted(set(SAMPLES) | set(_null_rows(ok)))
    res = p.outputs()
    if kernel != "base":
        _oracle_rows(res, d, ok, rows)
    else:
        for s in rows:
            c, h, l = (d[f][s] for f in ("close", "high", "low"))
            kc, kh, kl = (ok[f][s] for f in ("close", "high", "low"))
            sk, sd = pqo.stoch(h, l, c, 9, 3, 0, 3, 0, kh, kl, kc)
            jok = sk[1] & sd[1]
            for name, (rv, rk) in (("ema", pqo.ema(c, 30, kc)), ("atr", pqo.atr(h, l, c, 14, kh, kl, kc)), ("kdj_k", sk),
                                   ("kdj_d", sd), ("kdj_j", (np.where(jok, 3.0 * sk[0] - 2.0 * sd[0], np.nan), jok))):
                nbad, msg = T.compare(name, res[name][0][s], res[name][1][s], rv, rk)
                assert nbad == 0, f"symbol {s}: {msg}"
    if kernel == "extras":
        for s in rows:
            for name, (rv, rk) in expected(d, ok, s, DEFAULTS).items():
                if name in ("mom", "aroon_up", "aroon_down") + tuple(_outputs_of("dm")):
                    nbad, msg = T.compare(name, res[name][0][s], res[name][1][s], rv, rk)
                    assert nbad == 0, f"symbol {s}: {msg}"
    if kernel == "full":
        # the result columns of the chunk-edge symbols as one Arrow record batch: the host planes, nulls included
        sub = ["ema", "macd_hist", "rsi", "atr", "obv", "kdj_j", "midprice"]
        smask = sum(1 << N.OUTPUT_NAMES.index(n) for n in sub)
        rb = p.export_arrow(smask, ["S%04d" % s for s in range(S)])
        assert rb.num_columns == S * len(sub) and rb.num_rows == NB
        for s in SAMPLES + (2533,):
            for j, name in enumerate(sub):
                col = rb.column(s * len(sub) + j)
                assert rb.schema.names[s * len(sub) + j] == "S%04d_%s" % (s, name)
                gk = ~np.asarray(col.is_null())
                assert np.array_equal(gk, res[name][1][s]), (s, name)
                assert T.same_bits(np.asarray(col.to_numpy(zero_copy_only=False))[gk], res[name][0][s][gk]).all(), (s, name)
        del rb
    p.close(); ref.close()


def test_one_panel_through_a_sequence_of_null_patterns(pq, N, d):
    """The calls the benchmark repeats, on one panel: clean; nulls in chunk 2 only (the first null-bearing chunk is c > 0 on a
    panel that has never seen nulls); clean again; nulls in chunks 0 and 3 only; chunk 2's nulls with chunk 1 changed.  Each
    equals a fresh panel given the same columns, and a device-resident run() of the panel afterwards too."""
    params, mask = N.default_params(), (1 << N.N_SUITE_OUTPUTS) - 1
    steps = [_nulls(()), _nulls((2,)), _nulls(()), _nulls((0, 3)), _nulls((1, 2), variant=1)]
    p = pq.Panel(S, NB)
    for i, ok in enumerate(steps):
        refs, keep = _refs(pq, d, ok)
        p.run_columns(refs, params, threads=3)
        fresh = _staged(pq, d, ok, mask)
        fresh.run_host(params)
        _same(N, p, fresh, mask, f"step {i + 1}: run_columns")
        p.run(params)
        p.download()
        p.sync()
        _same(N, p, fresh, mask, f"step {i + 1}: run() after run_columns")
        if i in (1, 4):
            _oracle_rows(p.outputs(), d, ok, _null_rows(ok))
        fresh.close()
    p.close()


# ---- the same data as one Arrow record batch ---------------------------------------------------------------------------
F32_FROM = 2 * CS                                           # float32 closes in chunks 2 and 3


def _table(d, ok, lead=0):
    """`date`, then `{sym}_open` / close / high / low / volume per symbol: Float64 prices, Int64 volumes with their nulls,
    Float32 closes from symbol F32_FROM on; `lead` junk rows in front (for a sliced table)."""
    junk = np.full(lead, 7.0)
    cols, names = [pa.array(np.arange(-lead, NB, dtype=np.int64))], ["date"]
    for s in range(S):
        sym = "S%04d" % s
        cols.append(pa.array(np.concatenate([junk, d["open"][s]])))
        names.append(sym + "_open")
        for f in F:
            m = None if ok[f][s].all() else np.concatenate([np.zeros(lead, bool), ~ok[f][s]])
            v = np.concatenate([junk, d[f][s]])
            if f == "volume":
                v = v.astype(np.int64)
            elif f == "close" and s >= F32_FROM:
                v = v.astype(np.float32)
            cols.append(pa.array(v, mask=m))
            names.append("%s_%s" % (sym, f))
    return pa.table(cols, names=names)


def _column_map(table):
    sym = np.zeros(table.num_columns, dtype=np.int64)
    fld = np.full(table.num_columns, -1, dtype=np.int32)
    for i, name in enumerate(table.column_names):
        s, _, f = name.partition("_")
        if f in F:
            sym[i], fld[i] = int(s[1:]), F.index(f)
    return sym, fld


def _run_batch(N, p, params, table, threads, patch=None):
    """pqb_suite_run_record_batch over the table as one exported record batch; `patch(arr)` may edit the C struct first.
    Returns (rc, error text)."""
    rb = table.combine_chunks().to_batches()[0]
    arr, sch = N.ArrowArray(), N.ArrowSchema()
    rb._export_to_c(C.addressof(arr), C.addressof(sch))
    sym, fld = _column_map(table)
    undo = patch(arr) if patch else None
    try:
        rc = N.lib().pqb_suite_run_record_batch(p._h, C.byref(params), C.byref(arr), C.byref(sch), sym.ctypes.data, fld.ctypes.data,
                                                threads)
        return rc, N.lib().pqb_last_error().decode()
    finally:
        if undo:
            undo()
        from polars_quant_b200.wide import WidePanel
        WidePanel._release(arr, sch)


@pytest.fixture(scope="module")
def batch_case(d):
    """Item data of the record-batch tests: the item-2 null pattern, closes of chunks 2-3 rounded to float32."""
    ok = _nulls()
    dr = dict(d)
    dr["close"] = d["close"].copy()
    dr["close"][F32_FROM:] = d["close"][F32_FROM:].astype(np.float32).astype(np.float64)
    dr["volume"] = np.trunc(d["volume"])
    return dr, ok


def test_record_batch_over_four_chunks_with_casts_and_skipped_columns(pq, N, d, batch_case):
    """`date` and `{sym}_open` map to field -1, volumes are Int64 with nulls, closes of chunks 2-3 Float32 (cast on the intake
    threads: with one thread the GPU waits at every later chunk).  Equals the panel given the Float64 values; a WidePanel over
    the same table sliced by 3 rows (every column at an element / bit offset) equals it too."""
    from polars_quant_b200.wide import WidePanel
    params, mask = N.default_params(), (1 << N.N_SUITE_OUTPUTS) - 1
    dr, ok = batch_case
    ref = Reference(pq, N, dr, ok, params, mask)
    table = _table(dr, ok)
    assert table["S2000_close"].type == pa.float32() and table["S0100_close"].type == pa.float64()
    assert table["S0831_volume"].type == pa.int64() and table["S0832_volume"].null_count > 0
    p = pq.Panel(S, NB)
    for threads in (1, 0):
        rc, msg = _run_batch(N, p, params, table, threads)
        assert rc == 0, msg
        _same(N, p, ref.panel, mask, f"record batch threads={threads}")
    _oracle_rows(p.outputs(), dr, ok, sorted(set(SAMPLES) | set(_null_rows(ok))))
    p.close()
    del table
    lazy = WidePanel(_table(dr, ok, lead=3).slice(3)).suite(lazy=True)
    assert lazy.symbols == ["S%04d" % s for s in range(S)]
    for name in lazy.outputs:
        k = N.OUTPUT_NAMES.index(name)
        gv, gk = lazy.matrix(name)
        assert np.array_equal(gk, ref.panel.host_validity(k)), f"sliced table: {name} validity"
        assert T.same_bits(gv, ref.panel.host_output(k)).all(), f"sliced table: {name} values"
    del lazy
    ref.close()


def test_intake_errors_in_a_later_chunk(pq, N, d, batch_case):
    """A UTF-8 column mapped to a symbol of chunk 2 fails the call with PQB_ERR_UNSUPPORTED naming the dtype (chunks 0-1
    already on the GPU), and the next call on the panel equals a fresh panel.  A child shorter than the batch is refused
    with PQB_ERR_INVALID before anything is staged."""
    params, mask = N.default_params(), (1 << N.N_SUITE_OUTPUTS) - 1
    dr, ok = batch_case
    table = _table(dr, ok)
    i = table.column_names.index("S2000_high")
    bad = table.set_column(i, "S2000_high", pa.array(["%.3f" % x for x in dr["high"][2000]]))
    p = pq.Panel(S, NB)
    for threads in (1, 4):
        rc, msg = _run_batch(N, p, params, bad, threads)
        assert rc == -4 and "'u'" in msg, (rc, msg)
    rc, msg = _run_batch(N, p, params, table, 2)
    assert rc == 0, msg
    ref = Reference(pq, N, dr, ok, params, mask)
    _same(N, p, ref.panel, mask, "the call after an intake error")
    ref.close()
    before_in = p.host_field("close").copy()
    before_out = p.host_output(N.OUTPUT_NAMES.index("atr")).copy()
    j = table.column_names.index("S1700_low")
    other = pa.table([pa.array(np.roll(c.combine_chunks().to_numpy(zero_copy_only=False), 1)) if c.type == pa.float64() else c
                      for c in table.columns], names=table.column_names)

    def shorten(arr):
        child = arr.children[j].contents
        child.length = NB - 1
        def undo():
            child.length = NB
        return undo
    rc, msg = _run_batch(N, p, params, other, 2, patch=shorten)
    assert rc == -3 and "column %d" % j in msg, (rc, msg)
    assert np.array_equal(p.host_field("close").view(np.uint64), before_in.view(np.uint64))
    assert np.array_equal(p.host_output(N.OUTPUT_NAMES.index("atr")).view(np.uint64), before_out.view(np.uint64))
    p.close()


def _shard_nulls():
    """A flagged symbol in every fifth block: every chunk of every shard of a two-way split holds flagged and clean blocks."""
    ok = {f: np.ones((S, NB), bool) for f in F}
    for b in range(2, 80, 5):
        s = min(b * BLOCK + b % BLOCK, S - 1)
        if b % 2:
            ok["close"][s, 100 + 40 * b:110 + 40 * b] = False
        else:
            for f in F:
                ok[f][s, 4000 + b:] = False
    return ok


def test_same_device_shards_run_on_engines_of_their_own(pq, N, d):
    """`WidePanel.suite(devices=[0, 0])` and `[0, 0, 0]` on the 2,536-symbol table (two shards: 1,280 + 1,256 symbols, two
    chunks each), eager and lazy, equal the one-device table; every shard panel runs on an engine of its own."""
    from polars_quant_b200.shard import symbol_range
    from polars_quant_b200.wide import WidePanel
    ok = _shard_nulls()
    flagged = _flagged_blocks(ok)
    for g in range(2):
        lo, hi = symbol_range(S, 2, g)
        for c0 in range(lo, hi, CS):
            blocks = set(range(c0 // BLOCK, -(-min(c0 + CS, hi) // BLOCK)))
            assert blocks & flagged and blocks - flagged, (g, c0)
    wp = WidePanel(_table(d, ok))
    one = wp.suite()
    for devices in ([0, 0], [0, 0, 0]):
        many = wp.suite(devices=devices)
        assert many.column_names == one.column_names and many.equals(one), devices
        del many
        lazy = wp.suite(devices=devices, lazy=True)
        assert len(lazy._shards) == len(devices)
        assert len({sp.engine._h.value for sp, _, _ in lazy._shards}) == len(devices), "shards share an engine"
        assert lazy.table().equals(one), devices
        del lazy
