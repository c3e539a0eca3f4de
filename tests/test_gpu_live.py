"""Live panels on the B200: every pushed row equals, bit for bit (values where valid, and validity), the same row of one
pqb_suite_run over the concatenated history -- across push sizes that cross TMA stages, ring wraps and van Herk block ends,
ragged and multi-wave symbol counts, leading nulls that end in the history, inside a push or never, previews and refused
pushes."""
import numpy as np
import pyarrow as pa
import pytest

import synth
from oracle import pqo

pytestmark = pytest.mark.gpu

F = ("close", "high", "low", "volume")
PUSHES = (1, 2, 7, 8, 9, 31, 64)


def _data(S, N, seed=7):
    d = synth.ohlcv(S, N, seed=seed, sigma=0.02)
    return {f: np.ascontiguousarray(d[f]) for f in F}


def _mask(S, N, starts):
    ok = np.ones((S, N), dtype=bool)
    for s, a in starts.items():
        ok[s, :a] = False
    return ok


def _omask(ind):
    from polars_quant_b200 import _native as N
    m = (1 << N.N_SUITE_OUTPUTS) - 1 if ind & N.IND_ALL else 0
    if ind & sum(N.IND_EXTRA.values()):
        m |= ((1 << 43) - 1) & ~((1 << N.N_SUITE_OUTPUTS) - 1)
    if ind & N.IND_FASTK:
        m |= 1 << 43
    return m


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


def _full(pq, d, ok, n_bars, params, omask):
    p = _panel(pq, d, ok, n_bars, omask)
    res = {k: (v.copy(), m.copy()) for k, (v, m) in p.compute(params).items()}
    p.close()
    return res


def _rows(d, ok, t0, k):
    vals = [np.ascontiguousarray(d[f][:, t0:t0 + k].T) for f in F]
    valid = None if ok is None else np.ascontiguousarray(ok[:, t0:t0 + k].T)
    return vals, valid


def _same(got, full, t0, where=""):
    assert got, "no outputs"
    for name, (v, m) in got.items():
        fv, fm = full[name]
        k = v.shape[1]
        em = fm[:, t0:t0 + k]
        bad = np.argwhere(m != em)
        assert not len(bad), f"{where} {name}: validity differs at (symbol, row) {bad[:5].tolist()}"
        ev = fv[:, t0:t0 + k]
        diff = np.argwhere(m & (v.view(np.uint64) != ev.view(np.uint64)))
        assert not len(diff), f"{where} {name}: values differ at {diff[:5].tolist()}: {v[tuple(diff[0])]} vs {ev[tuple(diff[0])]}"


def _run_case(pq, N, S, T, params, ind, pushes=PUSHES, starts=None, max_push=64):
    total = T + sum(pushes)
    d = _data(S, total)
    ok = None if not starts else _mask(S, total, starts)
    om = _omask(ind)
    full = _full(pq, d, ok, total, params, om)
    hist = _panel(pq, d, ok, T, om)
    hist.compute(params)
    live = pq.LivePanel(hist, params, om, max_push)
    hist.close()
    t = T
    for k in pushes:
        vals, valid = _rows(d, ok, t, k)
        got = live.push(*vals, valid=valid)
        _same(got, full, t, f"push of {k} at bar {t}:")
        t += k
        assert live.bars == t
    live.close()


@pytest.fixture(scope="module")
def pq():
    import polars_quant_b200 as pq
    return pq


@pytest.fixture(scope="module")
def N():
    from polars_quant_b200 import _native as N
    return N


LEADS = {3: 50, 5: 305, 7: 10 ** 6, 40: 1, 99: 299}      # 3 / 40 / 99 start in the history, 5 inside the push of bars 303..309, 7 never


def test_default_suite_ragged_with_leading_nulls(pq, N):
    _run_case(pq, N, 100, 300, N.default_params(), N.IND_ALL, starts=LEADS)


def test_every_group_and_fastk(pq, N):
    ind = N.IND_ALL | sum(N.IND_EXTRA.values()) | N.IND_FASTK
    _run_case(pq, N, 70, 300, N.default_params(indicators=ind), ind, starts={s: a for s, a in LEADS.items() if s < 70})


def test_non_default_periods(pq, N):
    ind = N.IND_ALL | sum(N.IND_EXTRA.values())
    prm = N.default_params(indicators=ind, tema_period=1, willr_period=200, midprice_period=200, sma_period=3, bbands_period=5,
                           trima_period=4, kdj_fastk=5, kdj_slowk=2, kdj_slowd=4, macd_fast=5, macd_slow=3, macd_signal=2,
                           donchian_period=60, aroon_period=25, cci_period=7, mom_period=1, cmo_period=0)
    _run_case(pq, N, 33, 260, prm, ind, starts={2: 70})


def test_history_shorter_than_the_warm_up(pq, N):
    _run_case(pq, N, 40, 20, N.default_params(), N.IND_ALL, pushes=(64, 64, 1, 9), starts={1: 5, 2: 30})


def test_one_bar_history(pq, N):
    ind = N.IND_ALL | sum(N.IND_EXTRA.values())
    _run_case(pq, N, 35, 1, N.default_params(indicators=ind), ind, pushes=(1, 2, 7, 8, 9, 31, 64, 64))


def test_multi_wave(pq, N):
    _run_case(pq, N, 20000, 120, N.default_params(), N.IND_ALL, pushes=(1, 8, 9))


def test_against_the_oracle(pq, N):
    d = _data(3, 90)
    hist = _panel(pq, d, None, 50, (1 << 21) - 1)
    hist.compute()
    live = pq.LivePanel(hist, max_push_bars=40)
    got = live.push(*_rows(d, None, 50, 40)[0])
    for s in range(3):
        for name, ref in (("ema", pqo.ema(d["close"][s], 30)), ("rsi", pqo.rsi(d["close"][s], 14)),
                          ("willr", pqo.willr(d["high"][s], d["low"][s], d["close"][s], 14))):
            rv, rk = ref
            v, m = got[name]
            assert np.array_equal(m[s], rk[50:]), name
            assert np.array_equal(v[s][m[s]].view(np.uint64), rv[50:][rk[50:]].view(np.uint64)), name


def _hist_live(pq, d, T, ok=None, params=None, max_push=8):
    hist = _panel(pq, d, ok, T, (1 << 21) - 1)
    hist.compute(params)
    live = pq.LivePanel(hist, params, max_push_bars=max_push)
    hist.close()                                   # the live panel keeps no reference to its history
    return live


def test_preview_then_commit(pq, N):
    S, T = 50, 200
    d = _data(S, T + 3)
    full = _full(pq, d, None, T + 3, N.default_params(), (1 << 21) - 1)
    live = _hist_live(pq, d, T)
    made_up = [v * 1.37 for v in _rows(d, None, T, 1)[0]]
    live.push(*made_up, commit=False)
    assert live.bars == T
    live.push(*[v * 0.5 for v in made_up], commit=False)
    assert live.bars == T
    _same(live.push(*_rows(d, None, T, 1)[0]), full, T, "after previews:")
    assert live.bars == T + 1
    _same(live.push(*_rows(d, None, T + 1, 2)[0]), full, T + 1, "next push:")


def test_refused_pushes_leave_the_state_intact(pq, N):
    S, T = 40, 150
    d = _data(S, T + 4)
    starts = {6: 10 ** 4}                              # symbol 6 has no valid bar so far
    ok = _mask(S, T + 4, starts)
    ok[6, T + 2:] = True                               # ... and starts at bar T + 2
    full = _full(pq, d, ok, T + 4, N.default_params(), (1 << 21) - 1)
    live = _hist_live(pq, d, T, ok)
    vals, valid = _rows(d, ok, T, 1)
    bad = valid.copy()
    bad[0, 3] = False                                  # a null after symbol 3's start
    with pytest.raises(N.PqbError, match="PQB_ERR_UNSUPPORTED.*symbol 3 .*bar 150"):
        live.push(*vals, valid=bad)
    part = {f: valid.copy() for f in F}
    part["close"][0, 6] = True                         # symbol 6 starts with close valid and high / low null
    with pytest.raises(N.PqbError, match="PQB_ERR_UNSUPPORTED.*symbol 6 .*only some"):
        live.push(*vals, valid=part)
    too_many = [np.repeat(v, 9, axis=0) for v in vals]
    with pytest.raises(ValueError):
        live.push(*too_many)                           # (the Python check; the C ABI answers PQB_ERR_INVALID, below)
    import ctypes as C
    arrs = [np.ascontiguousarray(a) for a in too_many]
    rc = N.lib().pqb_live_push(live._h, C.c_int64(9), *(a.ctypes.data_as(C.c_void_p) for a in arrs), None, None, None, None, 1)
    assert rc == -3
    assert live.bars == T
    t = T
    for k in (1, 1, 2):
        v, m = _rows(d, ok, t, k)
        _same(live.push(*v, valid=m), full, t, f"after refusals, push at {t}:")
        t += k


def test_null_aware_history_is_refused(pq, N):
    S, T = 40, 100
    d = _data(S, T)
    ok = np.ones((S, T), dtype=bool)
    ok[4, 60] = False                                  # an interior null
    hist = _panel(pq, d, ok, T, (1 << 21) - 1)
    hist.compute()
    with pytest.raises(N.PqbError, match="PQB_ERR_UNSUPPORTED"):
        pq.LivePanel(hist)
    hist.close()


def test_two_live_panels_on_one_engine(pq, N):
    S, T = 64, 120
    da, db = _data(S, T + 20, seed=1), _data(S, T + 20, seed=2)
    fa = _full(pq, da, None, T + 20, N.default_params(), (1 << 21) - 1)
    fb = _full(pq, db, None, T + 20, N.default_params(), (1 << 21) - 1)
    la, lb = _hist_live(pq, da, T), _hist_live(pq, db, T)
    t = T
    for k in (1, 3, 8, 8):
        _same(la.push(*_rows(da, None, t, k)[0]), fa, t, "panel a:")
        _same(lb.push(*_rows(db, None, t, k)[0]), fb, t, "panel b:")
        t += k


def test_wide_live_matches_the_wide_suite(pq, N):
    from polars_quant_b200.wide import WidePanel
    S, T, K = 5, 80, 6
    d = _data(S, T + K)
    cols, names = [pa.array(np.arange(T + K, dtype=np.int64))], ["date"]
    for s in range(S):
        for f in F:
            v = d[f][s]
            mask = np.zeros(T + K, dtype=bool)
            if s == 2:
                mask[:T + 2] = True                    # a symbol listed during the pushed rows
            cols.append(pa.array(v, mask=mask))
            names.append("S%d_%s" % (s, f))
    table = pa.table(cols, names=names)
    hist, rows = table.slice(0, T), table.slice(T, K)
    head = WidePanel(hist).suite()
    wl = WidePanel(hist).live()
    tail = wl.push(rows)
    whole = WidePanel(table).suite()
    assert tail.column_names == whole.column_names == head.column_names
    got = pa.concat_tables([head, tail])
    for name in whole.column_names:
        assert got[name].combine_chunks().equals(whole[name].combine_chunks()), name
    with pytest.raises(NotImplementedError):
        WidePanel(hist).live(devices=[0, 1])
