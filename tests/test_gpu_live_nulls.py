"""Null-aware live panels on the B200 (LivePanel(..., nulls=True)): every pushed row equals, bit for bit where valid and
in validity exactly, the same row of Panel.compute over the concatenated history with the same bitmaps -- for histories
with halts, delistings, late listings and fields listed on different rows, for pushes with nulls anywhere -- and after
every push `voided` names exactly the (symbol, output) columns the new recompute turned all-null before the push."""
import numpy as np
import pyarrow as pa
import pytest

import synth
from oracle import pqo

pytestmark = pytest.mark.gpu

F = ("close", "high", "low", "volume")
PUSHES = (1, 2, 7, 8, 9, 31, 64)


@pytest.fixture(scope="module")
def pq():
    import polars_quant_b200 as pq
    return pq


@pytest.fixture(scope="module")
def N():
    from polars_quant_b200 import _native as N
    return N


def _data(S, n, seed=11):
    d = synth.ohlcv(S, n, seed=seed, sigma=0.02)
    return {f: np.ascontiguousarray(d[f]) for f in F}


def _ok(S, n):
    return {f: np.ones((S, n), dtype=bool) for f in F}


def _omask(N, ind):
    m = (1 << N.N_SUITE_OUTPUTS) - 1 if ind & N.IND_ALL else 0
    if ind & N.IND_FASTK:
        m |= 1 << N.OUTPUT_NAMES.index("fastk")
    return m


def _panel(pq, d, ok, n, omask):
    S = d["close"].shape[0]
    p = pq.Panel(S, n, outputs_mask=omask)
    for s in range(S):
        for f in F:
            m = ok[f][s, :n]
            p.set_column(s, f, d[f][s, :n], validity=None if m.all() else np.packbits(m, bitorder="little"))
    return p


def _full(pq, d, ok, n, params, omask):
    p = _panel(pq, d, ok, n, omask)
    res = {k: (v.copy(), m.copy()) for k, (v, m) in p.compute(params).items()}
    p.close()
    return res


def _rows(d, ok, t0, k):
    return [np.ascontiguousarray(d[f][:, t0:t0 + k].T) for f in F], {f: np.ascontiguousarray(ok[f][:, t0:t0 + k].T) for f in F}


def _same(got, full, t0, where):
    assert got, "no outputs"
    for name, (v, m) in got.items():
        fv, fm = full[name]
        k = v.shape[1]
        bad = np.argwhere(m != fm[:, t0:t0 + k])
        assert not len(bad), f"{where} {name}: validity differs at (symbol, row) {bad[:5].tolist()}"
        diff = np.argwhere(m & (v.view(np.uint64) != fv[:, t0:t0 + k].view(np.uint64)))
        assert not len(diff), f"{where} {name}: values differ at {diff[:5].tolist()}"


def _voided_ok(voided, prev, full, t, where):
    """voided == the columns valid somewhere before bar t in the previous recompute and nowhere in the new one; every
    other column's rows before t are unchanged"""
    for name, (v, m) in full.items():
        pv, pm = prev[name]
        was, now = pm[:, :t].any(axis=1), m[:, :t].any(axis=1)
        want = np.flatnonzero(was & ~now)
        got = voided.get(name, np.zeros(0, dtype=np.int64))
        assert np.array_equal(np.sort(got), want), f"{where} {name}: voided {got.tolist()}, expected {want.tolist()}"
        keep = np.setdiff1d(np.arange(m.shape[0]), want)
        assert np.array_equal(pm[keep, :t], m[keep, :t]), f"{where} {name}: earlier validity changed"
        assert np.array_equal(np.where(pm[keep, :t], pv[keep, :t], 0.0).view(np.uint64),
                              np.where(m[keep, :t], v[keep, :t], 0.0).view(np.uint64)), f"{where} {name}: earlier values changed"
    assert set(voided) <= set(full), voided


def _run(pq, N, d, ok, T, params, ind, pushes=PUSHES, max_push=64, check_voided=True):
    om = _omask(N, ind)
    hist = _panel(pq, d, ok, T, om)
    hist.compute(params)
    live = pq.LivePanel(hist, params, om, max_push, nulls=True)
    hist.close()
    prev = _full(pq, d, ok, T, params, om) if check_voided else None
    t = T
    for k in pushes:
        vals, valid = _rows(d, ok, t, k)
        got = live.push(*vals, valid=valid)
        full = _full(pq, d, ok, t + k, params, om)
        where = f"push of {k} at bar {t}:"
        _same(got, full, t, where)
        if check_voided:
            _voided_ok(live.voided, prev, full, t, where)
        prev = full
        t += k
        assert live.bars == t
    live.close()


def _real_universe(S, n, T):
    """halts in single fields and in all of them, delistings, late listings, fields listed on different rows, symbols
    that never trade, halts that fall into the pushes"""
    ok = _ok(S, n)
    ok["close"][1, 40:43] = False                          # close halted 3 bars in the history
    for f in F:
        ok[f][2, 100:103] = False                          # all fields halted
    ok["high"][3, 7] = False
    ok["low"][4, 250:252] = False
    ok["volume"][5, 20:40] = False                         # volume only (read by obv / ad)
    for f in F:
        ok[f][6, 280:] = False                             # delisted in the history
        ok[f][8, :303] = False                             # listed inside the push of bars 303 .. 309
        ok[f][9, :] = False                                # never trades
        ok[f][10, T + 40:] = False                         # delisted inside a push
    for f, a in zip(F, (10, 12, 14, 11)):
        ok[f][7, :a] = False                               # fields listed on different rows
    for f, a in zip(F, (T + 4, T + 5, T + 8, T + 4)):
        ok[f][12, :a] = False                              # ... inside one push, on different bars
    ok["close"][13, T] = False                             # first null after the listing: on a push's first bar
    ok["high"][14, T + 6] = False                          # ... on the last bar of the push of bars T+3 .. T+9
    ok["low"][15, T + 20:T + 23] = False
    for f in F:
        ok[f][16, T + 60:T + 63] = False                   # a halt crossing a push boundary
    for s in range(20, S, 9):                              # clustered halts
        ok["close"][s, 150 + s:153 + s] = False
    return ok


def test_halts_delistings_and_listings(pq, N):
    S, T = 70, 300
    d = _data(S, T + sum(PUSHES))
    _run(pq, N, d, _real_universe(S, T + sum(PUSHES), T), T, N.default_params(), N.IND_ALL)


@pytest.mark.parametrize("fields", [("close",), ("high",), ("low",), ("volume",), F])
def test_first_null_arrives_in_a_push(pq, N, fields):
    S, T, pushes = 35, 200, (8, 1, 64, 9)
    n = T + sum(pushes)
    d = _data(S, n, seed=3)
    ok = _ok(S, n)
    for i, bar in enumerate((T, T + 3, T + 7, T + 8, T + 9, T + 9 + 63)):   # first / middle / last bar of a push
        for f in fields:
            ok[f][2 * i, bar] = False
    ok["close"][30, :T + 2] = False                        # a symbol listed inside the first push
    _run(pq, N, d, ok, T, N.default_params(), N.IND_ALL, pushes)


def test_fastk_and_non_default_periods(pq, N):
    ind = N.IND_ALL | N.IND_FASTK
    prm = N.default_params(indicators=ind, tema_period=1, willr_period=200, midprice_period=200, sma_period=3, bbands_period=5,
                           trima_period=4, kdj_fastk=5, kdj_slowk=2, kdj_slowd=4, macd_fast=5, macd_slow=3, macd_signal=2)
    S, T = 35, 260
    n = T + sum(PUSHES)
    _run(pq, N, _data(S, n), _real_universe(S, n, T), T, prm, ind)


def test_donchian_fold(pq, N):
    ind = N.IND["midprice"] | N.IND["willr"] | N.IND_EXTRA["donchian"]
    prm = N.default_params(indicators=ind, midprice_period=20, donchian_period=20)
    S, T = 70, 300
    n = T + sum(PUSHES)
    om = (1 << N.OUTPUT_NAMES.index("midprice")) | (1 << N.OUTPUT_NAMES.index("willr")) | \
        (1 << N.OUTPUT_NAMES.index("donchian_upper")) | (1 << N.OUTPUT_NAMES.index("donchian_lower"))
    d, ok = _data(S, n), _real_universe(S, n, T)
    hist = _panel(pq, d, ok, T, om)
    hist.compute(prm)
    live = pq.LivePanel(hist, prm, om, 64, nulls=True)
    hist.close()
    prev, t = _full(pq, d, ok, T, prm, om), T
    for k in PUSHES:
        vals, valid = _rows(d, ok, t, k)
        got = live.push(*vals, valid=valid)
        assert {"donchian_upper", "donchian_lower"} <= set(got)
        full = _full(pq, d, ok, t + k, prm, om)
        _same(got, full, t, f"push at {t}:")
        _voided_ok(live.voided, prev, full, t, f"push at {t}:")
        prev, t = full, t + k


def test_ragged_clean_history(pq, N):
    S, T = 35, 150                                         # a clean history: the prime builds its validity from the starts
    n = T + sum(PUSHES)
    ok = _ok(S, n)
    for f in F:
        ok[f][4, :60] = False                              # leading nulls only: the history stays plain
    ok["close"][5, T + 30] = False
    _run(pq, N, _data(S, n), ok, T, N.default_params(), N.IND_ALL)


def test_multi_wave(pq, N):
    S, T, pushes = 20000, 120, (1, 8, 9)
    n = T + sum(pushes)
    rng = np.random.default_rng(5)
    ok = _ok(S, n)
    for s in rng.choice(S, S // 100, replace=False):       # 1 % of the symbols halted 3 bars in the history
        a = int(rng.integers(10, T - 3))
        for f in F:
            ok[f][s, a:a + 3] = False
    for t in range(T, n):                                  # 1 % of the symbols null in each pushed bar
        for s in rng.choice(S, S // 100, replace=False):
            ok["close"][s, t] = ok["high"][s, t] = False
    _run(pq, N, _data(S, n), ok, T, N.default_params(), N.IND_ALL, pushes, check_voided=False)


def test_preview_voids_then_clean_commit(pq, N):
    S, T = 40, 120
    d = _data(S, T + 3)
    ok = _ok(S, T + 3)
    params, om = N.default_params(), _omask(N, N.IND_ALL)
    hist = _panel(pq, d, ok, T, om)
    hist.compute(params)
    live = pq.LivePanel(hist, params, om, 8, nulls=True)
    hist.close()
    vals, valid = _rows(d, ok, T, 1)
    bad = {f: v.copy() for f, v in valid.items()}
    bad["close"][0, 3] = False
    live.push(*vals, valid=bad, commit=False)
    assert set(live.voided) == {"macd", "macd_signal", "macd_hist", "rsi", "willr"}
    assert all(list(v) == [3] for v in live.voided.values())
    assert live.bars == T
    got = live.push(*vals, valid=valid)
    assert live.voided == {}
    full = _full(pq, d, ok, T + 1, params, om)
    _same(got, full, T, "after the preview:")
    got = live.push(*_rows(d, ok, T + 1, 2)[0], valid=_rows(d, ok, T + 1, 2)[1])
    _same(got, _full(pq, d, ok, T + 3, params, om), T + 1, "next push:")


def test_against_the_oracle(pq, N):
    S, T, K = 3, 60, 40
    d = _data(S, T + K)
    ok = _ok(S, T + K)
    ok["close"][0, 30:33] = False                          # halted in the history
    ok["close"][1, T + 5:T + 7] = False                    # halted in the push
    hist = _panel(pq, d, ok, T, (1 << 21) - 1)
    hist.compute()
    live = pq.LivePanel(hist, max_push_bars=K, nulls=True)
    hist.close()
    vals, valid = _rows(d, ok, T, K)
    got = live.push(*vals, valid=valid)
    for s in range(S):
        c, cok = d["close"][s], ok["close"][s]
        for name, ref in (("ema", pqo.ema(c, 30, cok)), ("sma", pqo.sma(c, 30, cok))):
            rv, rk = ref
            v, m = got[name]
            assert np.array_equal(m[s], rk[T:]), (name, s)
            assert np.array_equal(v[s][m[s]].view(np.uint64), rv[T:][rk[T:]].view(np.uint64)), (name, s)
    assert not got["rsi"][1][:2].any()                     # rsi fails on a null close: all-null for symbols 0 and 1
    assert list(live.voided["rsi"]) == [1]                 # ... and this push did that to symbol 1
    rv, rk = pqo.rsi(d["close"][2], 14)
    assert np.array_equal(got["rsi"][1][2], rk[T:])
    assert np.array_equal(got["rsi"][0][2][rk[T:]].view(np.uint64), rv[T:][rk[T:]].view(np.uint64))


def test_optional_groups_are_refused(pq, N):
    S, T = 40, 100
    ind = N.IND_ALL | N.IND_EXTRA["mom"]
    hist = _panel(pq, _data(S, T), _ok(S, T), T, (1 << 21) - 1)
    hist.compute()
    with pytest.raises(N.PqbError, match="PQB_ERR_UNSUPPORTED"):
        pq.LivePanel(hist, N.default_params(indicators=ind), nulls=True)
    import ctypes as C
    out = C.c_void_p()
    assert N.lib().pqb_live_create_ex(hist._h, C.byref(N.default_params()), 0, 8, 2, C.byref(out)) == -3
    hist.close()


def test_wide_live_with_halts(pq, N):
    from polars_quant_b200.wide import WidePanel
    S, T, K = 6, 120, 9
    d = _data(S, T + K)
    ok = _ok(S, T + K)
    for f in F:
        ok[f][1, 50:53] = False                            # halted in the history
        ok[f][2, :T + 2] = False                           # listed during the pushed rows
    ok["close"][3, T + 4] = False                          # first null in the pushed rows: voids macd / rsi / willr
    ok["high"][4, T + 1] = False                           # voids willr / midprice
    cols, names = [pa.array(np.arange(T + K, dtype=np.int64))], ["date"]
    for s in range(S):
        for f in F:
            cols.append(pa.array(d[f][s], mask=~ok[f][s]))
            names.append("S%d_%s" % (s, f))
    table = pa.table(cols, names=names)
    hist, rows = table.slice(0, T), table.slice(T, K)
    head = WidePanel(hist).suite()
    wl = WidePanel(hist).live(nulls=True)
    tail = wl.push(rows)
    whole = WidePanel(table).suite()
    assert tail.column_names == whole.column_names == head.column_names
    changed = []
    for name in whole.column_names:
        w = whole[name].combine_chunks()
        assert tail[name].combine_chunks().equals(w.slice(T)), name
        if not head[name].combine_chunks().equals(w.slice(0, T)):
            changed.append(name)
            assert w.slice(0, T).null_count == T, name     # the only change to history: a column turned all-null
    assert sorted(wl.voided) == sorted(changed) and changed
