"""Live screens on the B200: after every push, the crossover signals, the MA cross and the info of a live panel equal
Panel.signals() / .ma_cross() / .info() of a recompute over the concatenated history -- signals exactly, info values
bit for bit where valid and validity exactly -- across push sizes, thresholds, MA kinds and periods, short histories,
late listings, partial suites, previews, null-aware panels and the wide-table layer."""
import ctypes as C

import numpy as np
import pyarrow as pa
import pytest

import synth

pytestmark = pytest.mark.gpu

F = ("close", "high", "low", "volume")
PUSHES = (1, 2, 7, 8, 9, 31, 64)
DERIVED = ("macd_cross", "kdj_cross", "rsi_cross")
SUITE = (1 << 21) - 1


@pytest.fixture(scope="module")
def pq():
    import polars_quant_b200 as pq
    return pq


@pytest.fixture(scope="module")
def N():
    from polars_quant_b200 import _native as N
    return N


def _data(S, n, seed=7):
    d = synth.ohlcv(S, n, seed=seed, sigma=0.02)
    return {f: np.ascontiguousarray(d[f]) for f in F}


def _mask(S, n, starts):
    ok = np.ones((S, n), dtype=bool)
    for s, a in starts.items():
        ok[s, :a] = False
    return ok


def _panel(pq, d, ok, n_bars, omask):
    S = d["close"].shape[0]
    p = pq.Panel(S, n_bars, outputs_mask=omask)
    if ok is None or ok[:, :n_bars].all():
        p.set_fields(**{f: d[f][:, :n_bars] for f in F})
    else:
        for s in range(S):
            bits = None if ok[s, :n_bars].all() else np.packbits(ok[s, :n_bars], bitorder="little")
            for f in F:
                p.set_column(s, f, d[f][s, :n_bars], validity=bits)
    return p


def _rows(d, ok, t0, k):
    vals = [np.ascontiguousarray(d[f][:, t0:t0 + k].T) for f in F]
    valid = None if ok is None else np.ascontiguousarray(ok[:, t0:t0 + k].T)
    return vals, valid


def _cross(a, b):
    out = np.zeros(a.shape, dtype=np.int8)
    with np.errstate(invalid="ignore"):
        out[:, 1:][(a[:, 1:] > b[:, 1:]) & (a[:, :-1] <= b[:, :-1])] = 1
        out[:, 1:][(a[:, 1:] < b[:, 1:]) & (a[:, :-1] >= b[:, :-1])] = -1
    return out


def _rule(res, oversold, overbought):
    """The header's rule, evaluated from validity on a recompute's outputs (a missing pair: zeros)."""
    val = lambda n: np.where(res[n][1], res[n][0], np.nan)
    S, T = res[next(iter(res))][0].shape
    z = np.zeros((S, T), dtype=np.int8)
    out = {"macd_cross": _cross(val("macd"), val("macd_signal")) if "macd" in res else z,
           "kdj_cross": _cross(val("kdj_k"), val("kdj_d")) if "kdj_k" in res else z}
    r = val("rsi") if "rsi" in res else np.full((S, T), np.nan)
    w = np.zeros((S, T), dtype=np.int8)
    with np.errstate(invalid="ignore"):
        w[:, 1:][(r[:, 1:] > oversold) & (r[:, :-1] <= oversold)] = 1
        w[:, 1:][(r[:, 1:] < overbought) & (r[:, :-1] >= overbought)] = -1
    out["rsi_cross"] = w
    return out


def _expected(pq, d, ok, n_bars, params, omask, scr, nulls):
    """the recompute's outputs and signals over bars [0, n_bars)"""
    p = _panel(pq, d, ok, n_bars, omask)
    res = {k: (v.copy(), m.copy()) for k, (v, m) in p.compute(params).items()}
    os_, ob = scr.get("oversold", 30.0), scr.get("overbought", 70.0)
    want = _rule(res, os_, ob)
    if not nulls:
        got = {k: v.copy() for k, v in p.signals(os_, ob).items()}
        for name in DERIVED:                           # (the panel function is the validity rule)
            assert np.array_equal(got[name], want[name]), name
        ma = scr.get("ma_cross", ("sma", 10, 20))
        if ma is not None:
            want["ma_cross"] = p.ma_cross(ma[1], ma[2], ma[0]).copy()
    p.close()
    return res, want


def _info(pq, d, ok, n_bars):
    p = _panel(pq, d, ok, n_bars, 1)
    p.upload()
    res = {k: (v.copy(), m.copy()) for k, (v, m) in p.info().items()}
    p.close()
    return res


def _same_info(got, want, where):
    for name, (v, m) in want.items():
        gv, gm = got[name]
        assert np.array_equal(gm, m), f"{where} info {name}: validity differs at {np.flatnonzero(gm != m)[:5]}"
        bad = np.flatnonzero(m & (gv.view(np.uint64) != v.view(np.uint64)))
        assert not len(bad), f"{where} info {name}: values differ at {bad[:5]}: {gv[bad[0]]} vs {v[bad[0]]}"
        assert np.isnan(gv[~gm]).all()


def _same_signals(got, want, t0, k, where, ma):
    names = DERIVED + (("ma_cross",) if ma else ())
    assert sorted(got) == sorted(names), (where, sorted(got))
    for name in names:
        e = want[name][:, t0:t0 + k]
        bad = np.argwhere(got[name] != e)
        assert not len(bad), f"{where} {name}: differs at (symbol, row) {bad[:5].tolist()}: {got[name][tuple(bad[0])]} vs {e[tuple(bad[0])]}"


def _run(pq, N, S, T, pushes=PUSHES, params=None, omask=SUITE, screen=None, starts=None, ok=None, d=None, nulls=False,
         max_push=64, info_every=True):
    scr = {} if screen is None else dict(screen)
    total = T + sum(pushes)
    d = _data(S, total) if d is None else d
    if ok is None and starts:
        ok = _mask(S, total, starts)
    params = params or N.default_params()
    _, want = _expected(pq, d, ok, total, params, omask, scr, nulls)
    info = scr.get("info", True)
    ma = scr.get("ma_cross", ("sma", 10, 20)) is not None
    hist = _panel(pq, d, ok, T, omask)
    hist.compute(params)
    live = pq.LivePanel(hist, params, omask, max_push, nulls=nulls, screen=scr or True)
    hist.close()
    if info:
        _same_info(live.info(), _info(pq, d, ok, T), "after create:")
    t = T
    total_sig = 0
    for i, k in enumerate(pushes):
        vals, valid = _rows(d, ok, t, k)
        live.push(*vals, valid=valid)
        where = f"push of {k} at bar {t}:"
        if nulls:                                      # (a null voids a whole column: the recompute ends at this push)
            want = _expected(pq, d, ok, t + k, params, omask, scr, nulls)[1]
        _same_signals(live.signals, want, t, k, where, ma)
        total_sig += sum(int((v != 0).sum()) for v in live.signals.values())
        t += k
        if info and (info_every or i == len(pushes) - 1):
            ref = _info(pq, d, ok, t)
            _same_info(live.last_info, ref, where)
            _same_info(live.info(), ref, where + " committed")
        assert live.bars == t
    live.close()
    return total_sig


LEADS = {3: 50, 5: 305, 7: 10 ** 6, 40: 1, 99: 299}      # 3 / 40 / 99 start in the history, 5 inside a push, 7 never


def test_default_screen_every_push_size_with_late_listings(pq, N):
    assert _run(pq, N, 100, 300, starts=LEADS) > 100


@pytest.mark.parametrize("kind", ["sma", "ema"])
@pytest.mark.parametrize("fast, slow", [(10, 20), (5, 60), (20, 10), (7, 7), (1, 3)])
def test_ma_kinds_and_periods(pq, N, kind, fast, slow):
    _run(pq, N, 40, 150, pushes=(1, 9, 64, 8), starts={2: 30, 5: 170, 9: 10 ** 6},
         screen=dict(ma_cross=(kind, fast, slow), info=False))


def test_ma_window_at_the_limit_and_past_it(pq, N):
    _run(pq, N, 33, 905, pushes=(1, 64), screen=dict(ma_cross=("sma", 3, 900), info=False), info_every=False)
    p = _panel(pq, _data(33, 50), None, 50, SUITE)
    p.compute()
    for bad, code in (((0, 4, 900), "PQB_ERR_UNSUPPORTED"), ((2, 10, 20), "PQB_ERR_UNSUPPORTED"), ((0, 0, 20), "PQB_ERR_INVALID"),
                      ((1, 10, -1), "PQB_ERR_INVALID")):
        assert N.ERR_NAMES[N.lib().pqb_ma_cross_run(p._h, *bad)] == code
        s = N.LiveScreen(30.0, 70.0, bad[0], bad[1], bad[2], 0)
        out = C.c_void_p()
        rc = N.lib().pqb_live_create_screen(p._h, C.byref(N.default_params()), 0, 8, 0, C.byref(s), C.byref(out))
        assert N.ERR_NAMES[rc] == code and not out.value, bad
    p.close()


def test_thresholds(pq, N):
    assert _run(pq, N, 64, 200, pushes=(1, 31, 64), screen=dict(oversold=45.0, overbought=55.0)) > 50


@pytest.mark.parametrize("T", [1, 5, 15])
def test_short_histories(pq, N, T):
    _run(pq, N, 35, T, pushes=(1, 2, 7, 8, 9, 31, 64), starts={1: 3, 4: 40}, screen=dict(ma_cross=("sma", 5, 60)))


def test_partial_suites_give_zero_signals(pq, N):
    no_macd = N.default_params(indicators=N.IND_ALL & ~N.IND["macd"])
    om = SUITE & ~(0b111 << 7)
    _run(pq, N, 40, 120, pushes=(1, 8, 9), params=no_macd, omask=om)
    no_kdj = N.default_params(indicators=N.IND_ALL & ~N.IND["kdj"])
    om = SUITE & ~(0b111 << 16)
    _run(pq, N, 40, 120, pushes=(1, 8, 9), params=no_kdj, omask=om)


def test_multi_wave(pq, N):
    _run(pq, N, 20000, 120, pushes=(1, 8, 9), starts={17: 125, 19999: 40})


def _made_up(d, t, k, scale):
    return [np.ascontiguousarray(d[f][:, t:t + k].T * scale) for f in F]


def test_preview_then_commit_and_preview_then_another_commit(pq, N):
    S, T = 50, 200
    d = _data(S, T + 6)
    scr = dict(ma_cross=("ema", 3, 8))
    _, want = _expected(pq, d, None, T + 6, N.default_params(), SUITE, scr, False)
    hist = _panel(pq, d, None, T, SUITE)
    hist.compute()
    live = pq.LivePanel(hist, max_push_bars=8, screen=scr)
    hist.close()
    committed = live.info()
    # a preview of other bars returns their screen ...
    alt = {f: d[f].copy() for f in F}
    for f in F:
        alt[f][:, T:T + 2] *= 1.05
    _, walt = _expected(pq, alt, None, T + 2, N.default_params(), SUITE, scr, False)
    live.push(*_made_up(d, T, 2, 1.05), commit=False)
    _same_signals(live.signals, walt, T, 2, "preview:", True)
    _same_info(live.last_info, _info(pq, alt, None, T + 2), "preview:")
    assert live.bars == T
    _same_info(live.info(), committed, "after the preview (committed):")
    # ... and keeps nothing: the real bars follow
    live.push(*_rows(d, None, T, 1)[0], commit=False)
    _same_signals(live.signals, want, T, 1, "preview of the real bar:", True)
    live.push(*_rows(d, None, T, 1)[0])
    _same_signals(live.signals, want, T, 1, "commit after previews:", True)
    live.push(*_made_up(d, T + 1, 3, 0.9), commit=False)
    live.push(*_rows(d, None, T + 1, 5)[0])
    _same_signals(live.signals, want, T + 1, 5, "a different commit after a preview:", True)
    _same_info(live.last_info, _info(pq, d, None, T + 6), "end:")


def test_null_aware_signals_with_halts_delistings_and_voiding(pq, N):
    S, T, pushes = 70, 200, (1, 2, 7, 8, 9, 31, 64)
    total = T + sum(pushes)
    rng = np.random.default_rng(5)
    ok = _mask(S, total, {3: 40, 8: 230, 11: 10 ** 6})
    for s in (4, 12, 30):
        ok[s, rng.integers(60, 190, 5)] = False          # halts in the history
    ok[20, 150:] = False                                 # delisted in the history
    ok[21, 260:] = False                                 # delisted during the pushes
    ok[25, T + 4] = False                                # a first halt inside a push: voids macd / rsi of symbol 25
    ok[26, T + 40:T + 43] = False
    d = _data(S, total)
    n = _run(pq, N, S, T, pushes=pushes, ok=ok, d=d, nulls=True, screen=dict(ma_cross=None, info=False))
    assert n > 100


def test_null_aware_refuses_ma_and_info(pq, N):
    S, T = 40, 100
    d = _data(S, T)
    ok = np.ones((S, T), dtype=bool)
    ok[4, 60] = False
    hist = _panel(pq, d, ok, T, SUITE)
    hist.compute()
    for scr in (True, dict(info=False), dict(ma_cross=None)):
        with pytest.raises(N.PqbError, match="PQB_ERR_UNSUPPORTED"):
            pq.LivePanel(hist, nulls=True, screen=scr)
    pq.LivePanel(hist, nulls=True, screen=dict(ma_cross=None, info=False)).close()
    hist.close()


@pytest.mark.parametrize("nulls", [False, True])
def test_outputs_are_the_same_with_and_without_a_screen(pq, N, nulls):
    S, T = 60, 150
    total = T + 40
    d = _data(S, total)
    ok = _mask(S, total, {2: 160, 6: 10 ** 6})
    if nulls:
        ok[9, 100] = False
        ok[10, T + 5] = False
    hist = _panel(pq, d, ok, T, SUITE)
    hist.compute()
    scr = dict(ma_cross=None, info=False) if nulls else True
    a = pq.LivePanel(hist, nulls=nulls)
    b = pq.LivePanel(hist, nulls=nulls, screen=scr)
    hist.close()
    assert b.state_bytes > a.state_bytes
    t = T
    for k in (1, 8, 31):
        vals, valid = _rows(d, ok, t, k)
        ra, rb = a.push(*vals, valid=valid), b.push(*vals, valid=valid)
        assert ra.keys() == rb.keys()
        for name in ra:
            assert ra[name][0].tobytes() == rb[name][0].tobytes() and np.array_equal(ra[name][1], rb[name][1]), name
        assert {k_: v.tolist() for k_, v in a.voided.items()} == {k_: v.tolist() for k_, v in b.voided.items()}
        t += k


def test_wide_live_info_and_signals(pq, N):
    from polars_quant_b200.wide import WidePanel
    S, T, K = 6, 90, 9
    d = _data(S, T + K)
    rng = np.random.default_rng(1)
    opens = rng.uniform(50, 150, (S, T + K))
    cols, names = [pa.array(np.arange(T + K, dtype=np.int64))], ["date"]
    for s in range(S):
        for f in ("open",) + F:
            mask = np.zeros(T + K, dtype=bool)
            if s == 2:
                mask[:T + 3] = True                      # listed during the pushed rows
            if f == "open" and s == 4:
                continue                                 # a symbol without an open column
            cols.append(pa.array(opens[s] if f == "open" else d[f][s], mask=mask))
            names.append("S%d_%s" % (s, f))
    table = pa.table(cols, names=names)
    wl = WidePanel(table.slice(0, T)).live(screen=True)
    assert wl.info().equals(WidePanel(table.slice(0, T)).info())
    t = T
    ok = np.ones((S, T + K), dtype=bool)
    ok[2, :T + 3] = False
    _, want = _expected(pq, d, ok, T + K, N.default_params(), SUITE, {}, False)
    for k in (4, 5):
        wl.push(table.slice(t, k))
        got = wl.signals
        assert got.column_names[0] == "date" and got.column("date").equals(table.slice(t, k).column("date"))
        for s in range(S):
            for name in DERIVED + ("ma_cross",):
                col = got.column("S%d_%s" % (s, name))
                assert col.type == pa.int8()
                assert np.array_equal(col.to_numpy(), want[name][s, t:t + k]), (s, name)
        t += k
        whole = WidePanel(table.slice(0, t)).info()
        mine = wl.info()
        assert mine.column_names == whole.column_names
        for name in whole.column_names:
            a, b = mine.column(name), whole.column(name)
            assert a.null_count == b.null_count and a.is_null().equals(b.is_null()), name
            if name == "symbol":
                assert a.equals(b)
            else:
                av, bv = a.to_numpy(zero_copy_only=False), b.to_numpy(zero_copy_only=False)
                m = ~np.asarray(a.is_null())
                assert np.array_equal(av[m].astype(np.float64).view(np.uint64), bv[m].astype(np.float64).view(np.uint64)), name
