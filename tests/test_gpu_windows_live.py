"""Live window panels on the B200 (WindowPanel.live -> WindowLive): every pushed row equals, bit for bit where valid and in
validity exactly, the same row of WindowPanel.compute over the concatenated history with the same bitmaps -- one- and
two-level windows, pushes across the two-level windows' block and segment boundaries, histories shorter than the longest
window, halts, delistings, listings and fields listed on different rows -- and after every push `voided` names exactly the
(symbol, line) columns the new recompute turned all-null before the push."""
import ctypes as C

import numpy as np
import pytest

import synth
from oracle import pqo

pytestmark = pytest.mark.gpu

F3 = ("close", "high", "low")
PUSHES = (1, 2, 7, 8, 9, 31, 64)
C5 = ((5, 9, 14, 60, 250), (5, 20, 55, 250), 14)


@pytest.fixture(scope="module")
def N():
    from polars_quant_b200 import _native as N
    return N


def _data(S, n, seed=11):
    d = synth.ohlcv(S, n, seed=seed, sigma=0.02)
    return {f: np.ascontiguousarray(d[f]) for f in F3}


def _ok(S, n):
    return {f: np.ones((S, n), dtype=bool) for f in F3}


def _panel(d, ok, n, kdj, ext, atr, sk=3, sd=3):
    from polars_quant_b200.windows import WindowPanel
    S = d["close"].shape[0]
    wp = WindowPanel(S, n, kdj=kdj, ext=ext, atr=atr, slowk_period=sk, slowd_period=sd)
    for s in range(S):
        for f in F3:
            m = ok[f][s, :n]
            wp.panel.set_column(s, f, d[f][s, :n], validity=None if m.all() else np.packbits(m, bitorder="little"))
    return wp


def _full(d, ok, n, win):
    wp = _panel(d, ok, n, *win)
    res = {k: (v.copy(), m.copy()) for k, (v, m) in wp.compute().items()}
    wp.close()
    return res


def _rows(d, ok, t0, k):
    return [np.ascontiguousarray(d[f][:, t0:t0 + k].T) for f in F3], {f: np.ascontiguousarray(ok[f][:, t0:t0 + k].T) for f in F3}


def _same(got, full, t0, where):
    assert set(got) == set(full), (sorted(got), sorted(full))
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


def _run(d, ok, T, win, pushes=PUSHES, max_push=64, check_voided=True):
    hist = _panel(d, ok, T, *win)
    hist.compute()
    live = hist.live(max_push)
    hist.close()                                           # the live panel keeps no reference to it
    prev = _full(d, ok, T, win) if check_voided else None
    t = T
    for k in pushes:
        vals, valid = _rows(d, ok, t, k)
        got = live.push(*vals, valid=valid)
        full = _full(d, ok, t + k, win)
        where = f"push of {k} at bar {t}:"
        _same(got, full, t, where)
        if check_voided:
            _voided_ok(live.voided, prev, full, t, where)
        prev = full
        t += k
        assert live.bars == t
    assert live.last_push_ms() > 0.0 and live.state_bytes > 0
    live.close()


def _universe(S, n, T):
    """halts in single fields and in all of them, delistings, listings inside a push, never-listed symbols, fields listed on
    different rows, first nulls inside the pushes"""
    ok = _ok(S, n)
    ok["close"][1 % S, 40:43] = False                      # close halted in the history: WILLR dies
    if S > 2:
        for f in F3:
            ok[f][2, 100:103] = False                      # all fields halted
    if S > 16:
        ok["high"][3, 7] = False
        ok["low"][4, T - 2:T] = False                      # halted on the history's last bars
        for f in F3:
            ok[f][6, T // 2:] = False                      # delisted in the history
            ok[f][8, :T + 3] = False                       # listed inside the first pushes
            ok[f][9, :] = False                            # never trades
            ok[f][10, T + 40:] = False                     # delisted inside a push
        for f, a in zip(F3, (10, 12, 14)):
            ok[f][7, :a] = False                           # fields listed on different rows
        for f, a in zip(F3, (T + 4, T + 5, T + 8)):
            ok[f][11, :a] = False                          # ... inside one push, on different bars
        ok["close"][12, T] = False                         # a first null on a push's first bar
        ok["high"][13, T + 9] = False
        ok["low"][14, T + 20:T + 23] = False
        for f in F3:
            ok[f][15, T + 60:T + 63] = False               # a halt crossing a push boundary
        for s in range(20, S, 9):                          # clustered close halts
            ok["close"][s, 20 + s % 50:23 + s % 50] = False
    return ok


WINDOWS = {
    "one_level": ((5, 9, 14), (5, 20, 32), 14),
    "two_level": ((33, 60), (128, 250), 0),
    "config5": C5,
    "atr_alone": ((), (), 14),
    "one_unit": ((), (33,), 0),
    "twelve_units": ((1, 5, 9, 33, 60, 250), (5, 20, 33, 128, 250), 14),
}


@pytest.mark.parametrize("name", sorted(WINDOWS))
def test_windows_with_halts_and_delistings(N, name):
    S, T = 70, 301                                         # (a history length that is not a multiple of 8)
    n = T + sum(PUSHES)
    _run(_data(S, n), _universe(S, n, T), T, WINDOWS[name])


@pytest.mark.parametrize("sk,sd", [(1, 64), (64, 1)])
def test_smoothing_periods(N, sk, sd):
    S, T = 40, 205
    n = T + sum(PUSHES)
    _run(_data(S, n, seed=4), _universe(S, n, T), T, ((5, 33, 60), (9,), 0, sk, sd))


def test_history_shorter_than_the_longest_window(N):
    S, T, pushes = 35, 13, (1, 2, 7, 8, 9, 31, 64, 64, 64, 64)   # the 250-bar windows' first blocks end inside the pushes
    n = T + sum(pushes)
    ok = _ok(S, n)
    ok["close"][3, T + 100:T + 102] = False
    for f in F3:
        ok[f][4, :T + 50] = False                          # listed long after the history
    ok["high"][5, T + 255] = False
    _run(_data(S, n, seed=7), ok, T, ((9, 60, 250), (33, 250), 14), pushes)


@pytest.mark.parametrize("p", [33, 60, 128, 250])
def test_pushes_across_block_and_segment_boundaries(N, p):
    # two-level window p: blocks of p bars, segments of b = 8 (16 from 128 on).  The history ends one bar before block 3;
    # single-bar pushes land on t = 3p - 1, 3p, 3p + 1 and on segment edges, a 64-bar push crosses two blocks of a 33-bar window
    b = 16 if p >= 128 else 8
    S, T = 33, 3 * p - 1
    pushes = (1, 1, 1, b - 3, 1, 1, 1, 64, b, 1, 64)
    n = T + sum(pushes)
    ok = _ok(S, n)
    ok["high"][2, T + 1] = False                           # a first null on the block's first bar
    ok["low"][3, T + b] = False
    ok["close"][4, T + 2] = False
    _run(_data(S, n, seed=p), ok, T, ((p,), (p,), 14), pushes)


@pytest.mark.parametrize("field", F3)
def test_first_null_on_the_first_middle_and_last_bar_of_a_push(N, field):
    S, T, pushes = 35, 200, (8, 1, 64, 9)
    n = T + sum(pushes)
    ok = _ok(S, n)
    for i, bar in enumerate((T, T + 3, T + 7, T + 8, T + 9, T + 9 + 63)):
        ok[field][2 * i, bar] = False
    ok[field][30, :T + 2] = False                          # this field listed inside the first push
    _run(_data(S, n, seed=3), ok, T, ((9, 60), (20, 55), 14), pushes)


@pytest.mark.parametrize("S", [1, 33, 70])
def test_ragged_symbol_counts(N, S):
    T = 150
    n = T + sum(PUSHES)
    _run(_data(S, n, seed=S), _universe(S, n, T), T, ((9, 33), (5, 128), 14))


def test_multi_wave(N):
    S, T, pushes = 10000, 300, (1, 8, 64)
    n = T + sum(pushes)
    rng = np.random.default_rng(5)
    ok = _ok(S, n)
    for s in rng.choice(S, S // 100, replace=False):       # 1 % of the symbols halted 3 bars in the history
        a = int(rng.integers(10, T - 3))
        for f in F3:
            ok[f][s, a:a + 3] = False
    for t in range(T, n):                                  # 1 % of the symbols null in each pushed bar
        for s in rng.choice(S, S // 100, replace=False):
            ok["close"][s, t] = ok["high"][s, t] = False
    _run(_data(S, n), ok, T, C5, pushes, check_voided=False)


def test_preview_voids_then_clean_commit(N):
    S, T, win = 40, 120, ((9,), (20, 33), 14)
    d, ok = _data(S, T + 3), _ok(S, T + 3)
    hist = _panel(d, ok, T, *win)
    hist.compute()
    live = hist.live(8)
    hist.close()
    vals, valid = _rows(d, ok, T, 1)
    bad = {f: v.copy() for f, v in valid.items()}
    bad["close"][0, 3] = False
    bad["high"][0, 5] = False
    live.push(*vals, valid=bad, commit=False)
    want = {"willr_20": [3, 5], "willr_33": [3, 5]}           # willr: close or high; midprice / Donchian: high only
    for line in ("midprice", "donchian_upper", "donchian_lower"):
        want.update({"%s_20" % line: [5], "%s_33" % line: [5]})
    assert {k: list(v) for k, v in live.voided.items()} == want
    assert live.bars == T
    got = live.push(*vals, valid=valid)
    assert live.voided == {}
    _same(got, _full(d, ok, T + 1, win), T, "after the preview:")
    vals, valid = _rows(d, ok, T + 1, 2)
    _same(live.push(*vals, valid=valid), _full(d, ok, T + 3, win), T + 1, "next push:")


def test_two_live_panels_on_one_engine(N):
    S, T = 45, 140
    n = T + 40
    d, ok = _data(S, n, seed=9), _universe(S, n, T)
    wa, wb = ((9, 33), (5, 60), 14), ((14,), (250,), 0)
    la, lb = [], []
    for win, out in ((wa, la), (wb, lb)):
        h = _panel(d, ok, T, *win)
        h.compute()
        out.append(h.live(16))
        h.close()
    t = T
    for k in (3, 16, 1, 9, 11):
        vals, valid = _rows(d, ok, t, k)
        ga = la[0].push(*vals, valid=valid)
        gb = lb[0].push(*vals, valid=valid)
        _same(ga, _full(d, ok, t + k, wa), t, f"panel a at {t}:")
        _same(gb, _full(d, ok, t + k, wb), t, f"panel b at {t}:")
        t += k
    la[0].close()
    lb[0].close()


def test_create_leaves_the_window_panel_alone(N):
    S, T, win = 40, 100, ((9, 60), (20, 128), 14)
    d, ok = _data(S, T + 64), _universe(S, T + 64, T)
    wp = _panel(d, ok, T, *win)
    before = {k: (v.copy(), m.copy()) for k, (v, m) in wp.compute().items()}
    live = wp.live(16)
    wp.panel.download()
    wp.panel.sync()
    after = {name: (wp.panel.host_output(k), wp.panel.host_validity(k)) for k, name in wp.names().items()}
    for name, (v, m) in before.items():
        assert np.array_equal(m, after[name][1]), name
        assert np.array_equal(np.where(m, v, 0.0).view(np.uint64), np.where(m, after[name][0], 0.0).view(np.uint64)), name
    wp.close()
    vals, valid = _rows(d, ok, T, 9)
    _same(live.push(*vals, valid=valid), _full(d, ok, T + 9, win), T, "after closing the window panel:")
    live.close()


def test_against_the_oracle(N):
    S, T, K = 4, 90, 40
    d, ok = _data(S, T + K, seed=2), _ok(S, T + K)
    ok["close"][0, 30:33] = False                          # halted in the history
    ok["high"][1, T + 5:T + 7] = False                     # halted in the push
    for f in F3:
        ok[f][2, :T + 10] = False                          # listed inside the push
    win = ((9,), (20,), 14)
    hist = _panel(d, ok, T, *win)
    hist.compute()
    live = hist.live(K)
    hist.close()
    vals, valid = _rows(d, ok, T, K)
    got = live.push(*vals, valid=valid)
    for s in range(S):
        h, l, c = (d[f][s] for f in ("high", "low", "close"))
        kh, kl, kc = (ok[f][s].astype(np.uint8) for f in ("high", "low", "close"))
        K_, D_ = pqo.stoch(h, l, c, 9, 3, 0, 3, 0, kh, kl, kc)
        refs = {"kdj_k_9": K_, "kdj_d_9": D_, "atr_14": pqo.atr(h, l, c, 14, kh, kl, kc)}
        hl = ok["high"][s] & ok["low"][s]
        a = int(np.argmax(hl))
        if s != 1:                                          # (symbol 1: flagged in high, its midprice / willr are all-null)
            mv, mk = pqo.midprice(h[a:], l[a:], 20)
            refs["midprice_20"] = (np.r_[np.full(a, np.nan), mv], np.r_[np.zeros(a, bool), mk])
        if s == 3:
            refs["willr_20"] = pqo.willr(h, l, c, 20)
        for name, (rv, rk) in refs.items():
            v, m = got[name]
            assert np.array_equal(m[s], rk[T:]), (name, s)
            assert np.array_equal(v[s][m[s]].view(np.uint64), rv[T:][rk[T:]].view(np.uint64)), (name, s)
    assert not got["midprice_20"][1][1].any() and not got["willr_20"][1][0].any()
    assert list(live.voided["midprice_20"]) == [1] and list(live.voided["willr_20"]) == [1]
    live.close()


def test_refusals(N, monkeypatch):
    from polars_quant_b200.windows import WindowPanel
    L = N.lib()
    S, T, win = 40, 100, ((9,), (33,), 14)
    d, ok = _data(S, T + 8), _ok(S, T + 8)
    out = C.c_void_p()
    cold = WindowPanel(S, T, kdj=(9,), ext=(33,), atr=14)  # inputs never uploaded
    assert L.pqb_windows_live_create(cold._h, 8, C.byref(out)) == -3 and not out.value
    cold.close()
    wp = _panel(d, ok, T, *win)
    wp.compute()
    for bad in (0, -1, (1 << 20) + 1):
        assert L.pqb_windows_live_create(wp._h, bad, C.byref(out)) == -3 and not out.value
    assert L.pqb_windows_live_create(None, 8, C.byref(out)) == -3
    live = wp.live(8)
    wp.close()
    vals, valid = _rows(d, ok, T, 8)
    p = [v.ctypes.data_as(C.c_void_p) for v in vals]
    assert L.pqb_windows_live_push(live._h, 9, *p, None, None, None, 1) == -3          # more than max_push_bars
    assert L.pqb_windows_live_push(live._h, -1, *p, None, None, None, 1) == -3
    assert L.pqb_windows_live_push(live._h, 2, p[0], None, p[2], None, None, None, 1) == -3   # a NULL field
    assert L.pqb_windows_live_push(live._h, 0, None, None, None, None, None, None, 1) == 0    # k = 0: a no-op
    assert live.bars == T
    got = live.push(*vals, valid=valid)                    # the refused pushes changed nothing
    _same(got, _full(d, ok, T + 8, win), T, "after the refusals:")
    live.close()
    # a plan without shared memory for the walk's validity words (one-level KDJ(425), smoothings 3 / 4: 232,320 bytes)
    monkeypatch.setenv("PQB_WIN_SMEM_MAX", "1000")
    big = WindowPanel(S, T, kdj=(425,), ext=(), atr=0, slowk_period=3, slowd_period=4)
    big.fill_synthetic()
    assert L.pqb_windows_live_create(big._h, 8, C.byref(out)) == -4 and not out.value
    big.close()
