"""Live candle panels on the B200 (CandlePanel.live -> CandleLive): every pushed row equals the same row of
CandlePanel.run_host over the concatenated history -- Int32 patterns exactly, prices bit for bit where valid and their
validity exactly -- on the golden panel split at many bars, histories shorter than the 4-bar lookback, both kernel
specialisations, prices with nulls, refused pushes, previews and a multi-wave panel; spot checks against the C oracle."""
import ctypes as C
from pathlib import Path

import numpy as np
import pytest

from polars_quant_b200 import _native as N
from polars_quant_b200 import candles

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parents[1]
F4 = ("open", "high", "low", "close")
PUSHES = (1, 2, 3, 4, 5, 7, 8, 31, 64)
ALL_PATTERNS = (1 << N.N_PATTERNS) - 1
PRICES = 0b01111                                           # the four price transforms (bop refuses nulls)


@pytest.fixture(scope="module")
def g():
    return np.load(ROOT / "tests" / "golden" / "candle_golden.npz")


def _golden(g):
    return {f: np.ascontiguousarray(g[f]) for f in F4}


def _params(patterns=ALL_PATTERNS, prices=(1 << N.N_PRICES) - 1, penetration=None):
    return candles.default_params(patterns=patterns, prices=prices, penetration=penetration)


def _panel(d, n, prm, ok=None):
    S = d["open"].shape[0]
    p = candles.CandlePanel(S, n, patterns_mask=prm.patterns, prices_mask=prm.prices)
    p.set_fields(*(d[f][:, :n] for f in F4), validity=None if ok is None else {i: ok[f][:, :n] for i, f in enumerate(F4)})
    return p


def _full(d, n, prm, ok=None):
    """the recompute over the first n bars: ({pattern name: Int32 [S, n]}, {price name: (values, validity)})"""
    p = _panel(d, n, prm, ok)
    p.run_host(prm)
    names = candles.pattern_names()
    pats = {names[k]: p.pattern(k).copy() for k in range(N.N_PATTERNS) if prm.patterns >> k & 1}
    prices = {}
    for q in range(N.N_PRICES):
        if prm.prices >> q & 1:
            v, m = p.price(q)
            prices[N.PRICE_NAMES[q]] = (v.copy(), m.copy())
    p.close()
    return pats, prices


def _rows(d, t, k, ok=None, fields=F4):
    vals = {f: (np.ascontiguousarray(d[f][:, t:t + k].T) if f in fields else None) for f in F4}
    valid = None if ok is None else {f: np.ascontiguousarray(ok[f][:, t:t + k].T) for f in fields}
    return vals, valid


def _same(got, full, t0, where):
    pats, prices = got
    fp, fpr = full
    assert set(pats) == set(fp) and set(prices) == set(fpr), (sorted(pats), sorted(prices))
    hits = 0
    for name, v in pats.items():
        want = fp[name][:, t0:t0 + v.shape[1]]
        bad = np.argwhere(v != want)
        assert not len(bad), f"{where} {name}: differs at (symbol, row) {bad[:5].tolist()}"
        hits += int((v != 0).sum())
    for name, (v, m) in prices.items():
        fv, fm = fpr[name]
        k = v.shape[1]
        bad = np.argwhere(m != fm[:, t0:t0 + k])
        assert not len(bad), f"{where} {name}: validity differs at {bad[:5].tolist()}"
        diff = np.argwhere(m & (v.view(np.uint64) != fv[:, t0:t0 + k].view(np.uint64)))
        assert not len(diff), f"{where} {name}: values differ at {diff[:5].tolist()}"
        assert np.isnan(v[~m]).all(), f"{where} {name}: a value under a null is not NaN"
    return hits


def _run(d, T, prm, pushes=PUSHES, ok=None, fields=F4, max_push=64):
    hist = _panel(d, T, prm, ok)
    hist.run_host(prm)
    live = hist.live(prm, max_push)
    hist.close()                                           # the live panel keeps no reference to it
    t, hits = T, 0
    for k in pushes:
        vals, valid = _rows(d, t, k, ok, fields)
        got = live.push(**vals, valid=valid)
        hits += _same(got, _full(d, t + k, prm, ok), t, f"push of {k} at bar {t}:")
        t += k
        assert live.bars == t
    assert live.last_push_ms() > 0.0
    live.close()
    return hits


SUBSET = ("cdl3outside", "cdlbreakaway", "cdldarkcloudcover", "cdldoji", "cdlengulfing", "cdleveningstar", "cdlhammer",
          "cdlladderbottom", "cdlmathold", "cdlmorningdojistar", "cdlpiercing", "cdlrisefall3methods")


def _spec(g, name):
    """the ALL kernel (61 patterns) and the masked one, at the default penetration and at the golden file's"""
    pen = float(g["penetration_value"]) if name.endswith("_pen") else None
    if name.startswith("all"):
        return _params(penetration=pen)
    names = candles.pattern_names()
    return _params(patterns=sum(1 << names.index(x) for x in SUBSET), prices=0b10110, penetration=pen)


@pytest.mark.parametrize("spec", ["all", "all_pen", "subset", "subset_pen"])
@pytest.mark.parametrize("T", [6, 100, 255, 256, 275])
def test_golden_panel_split_at_many_bars(g, T, spec):
    hits = _run(_golden(g), T, _spec(g, spec))
    assert hits > 500


def test_live_rows_are_the_golden_vectors(g):
    d, T = _golden(g), 200
    hist = _panel(d, T, _params())
    hist.run_host()
    live = hist.live(max_push_bars=64)
    hist.close()
    names = [str(n) for n in g["names"]]
    for t in range(T, 400, 50):
        vals, _ = _rows(d, t, 50)
        pats, prices = live.push(**vals)
        for k, n in enumerate(names):
            assert np.array_equal(pats[n], g["patterns"][k][:, t:t + 50].astype(np.int32)), (n, t)
        for q, n in enumerate(N.PRICE_NAMES):
            assert prices[n][1].all() and np.array_equal(prices[n][0].view(np.uint64), g["prices"][q][:, t:t + 50].view(np.uint64))
    live.close()


@pytest.mark.parametrize("spec", ["all", "subset_pen"])
@pytest.mark.parametrize("T", [1, 2, 3, 4, 5])
def test_history_shorter_than_the_lookback(g, T, spec):
    _run(_golden(g), T, _spec(g, spec), pushes=(1, 1, 2, 3, 4, 5, 64))


def _null_universe(S, n, T, seed=3):
    rng = np.random.default_rng(seed)
    ok = {f: rng.random((S, n)) > 0.05 for f in F4}        # 5 % nulls everywhere, history and pushes
    for f in F4:
        ok[f][0, :] = False                                # a symbol that never trades
        ok[f][1, T:] = False                               # delisted at the end of the history
        ok[f][2, :T + 3] = False                           # listed inside the first push
        ok[f][3, :] = True                                 # a clean one
    ok["high"][4, T - 1] = False                           # a null on the history's last bar
    ok["close"][5, T] = False                              # ... and on the first pushed bar
    return ok


@pytest.mark.parametrize("prices", [PRICES, 1 << 0, 1 << 1, 1 << 2, 1 << 3])
def test_prices_only_with_nulls(g, prices):
    d, T = _golden(g), 150
    ok = _null_universe(d["open"].shape[0], 400, T)
    prm = _params(patterns=0, prices=prices)
    _run(d, T, prm, ok=ok)


def test_unread_fields_may_be_none(g):
    d, T = _golden(g), 120
    ok = _null_universe(d["open"].shape[0], 400, T, seed=5)
    _run(d, T, _params(patterns=0, prices=1 << 1), ok=ok, fields=("high", "low"))            # medprice: high / low
    _run(d, T, _params(patterns=0, prices=0b01100), ok=ok, fields=("high", "low", "close"))  # typprice, wclprice


def test_refusals(g):
    L = N.lib()
    d, T = _golden(g), 100
    S = d["open"].shape[0]
    prm = _params()
    out = C.c_void_p()
    cold = candles.CandlePanel(S, T)                       # inputs never on the device
    cold.set_fields(*(d[f][:, :T] for f in F4))
    assert L.pqb_candles_live_create(cold._h, C.byref(prm), 8, C.byref(out)) == -3 and not out.value
    cold.run_host()
    for bad in (0, -1, (1 << 20) + 1):
        assert L.pqb_candles_live_create(cold._h, C.byref(prm), bad, C.byref(out)) == -3 and not out.value
    wide = _params()
    wide.patterns = 1 << N.N_PATTERNS
    assert L.pqb_candles_live_create(cold._h, C.byref(wide), 8, C.byref(out)) == -3 and not out.value
    cold.close()
    # a history with nulls: patterns and bop are refused at create, the price transforms are not
    ok = {f: np.ones((S, 400), dtype=bool) for f in F4}
    ok["low"][9, 40] = False
    nh = _panel(d, T, _params(), ok)
    nh.run_host(_params(patterns=0, prices=PRICES))
    for p in (_params(), _params(patterns=1, prices=0), _params(patterns=0, prices=1 << 4)):
        with pytest.raises(N.PqbError) as e:
            nh.live(p)
        assert e.value.code == -5                          # PQB_ERR_NULLS
    nh.live(_params(patterns=0, prices=PRICES)).close()
    nh.close()
    # a null in a pushed bar: refused with the symbol, bar and field named, and nothing changes
    hist = _panel(d, T, prm)
    hist.run_host()
    live = hist.live(prm, 8)
    hist.close()
    vals, _ = _rows(d, T, 8)
    bad = {f: np.ones((8, S), dtype=bool) for f in F4}
    bad["close"][3, 17] = False
    with pytest.raises(N.PqbError) as e:
        live.push(**vals, valid=bad)
    assert e.value.code == -5 and "close of symbol 17" in str(e.value) and "bar %d" % (T + 3) in str(e.value)
    assert live.bars == T
    p = [vals[f].ctypes.data_as(C.c_void_p) for f in F4]
    assert L.pqb_candles_live_push(live._h, 9, *p, None, None, None, None, 1) == -3          # more than max_push_bars
    assert L.pqb_candles_live_push(live._h, -1, *p, None, None, None, None, 1) == -3
    assert L.pqb_candles_live_push(live._h, 2, p[0], None, p[2], p[3], None, None, None, None, 1) == -3   # a NULL field
    assert L.pqb_candles_live_push(live._h, 0, *([None] * 8), 1) == 0                        # k = 0: a no-op
    assert live.bars == T
    _same(live.push(**vals), _full(d, T + 8, prm), T, "after the refusals:")
    vals, _ = _rows(d, T + 8, 1)
    _same(live.push(**vals), _full(d, T + 9, prm), T + 8, "next push:")
    live.close()
    # bop alone refuses nulls in pushes too
    bop = _params(patterns=0, prices=1 << 4)
    hist = _panel(d, T, bop)
    hist.run_host(bop)
    live = hist.live(bop, 8)
    hist.close()
    vals, _ = _rows(d, T, 1)
    one = {f: np.ones((1, S), dtype=bool) for f in F4}
    one["open"][0, 0] = False
    with pytest.raises(N.PqbError, match="open of symbol 0"):
        live.push(**vals, valid=one)
    _same(live.push(**vals), _full(d, T + 1, bop), T, "bop after a refusal:")
    live.close()


def test_preview_then_a_different_committed_bar(g):
    d, T = _golden(g), 180
    prm = _params()
    hist = _panel(d, T, prm)
    hist.run_host()
    live = hist.live(prm, 8)
    hist.close()
    other = {f: d[f].copy() for f in F4}                   # bar T of a shuffled symbol order: a different bar
    perm = np.random.default_rng(1).permutation(d["open"].shape[0])
    for f in F4:
        other[f][:, T] = d[f][perm, T + 30]
    vals, _ = _rows(other, T, 1)
    _same(live.push(**vals, commit=False), _full(other, T + 1, prm), T, "preview:")
    assert live.bars == T
    _same(live.push(**vals, commit=False), _full(other, T + 1, prm), T, "the same preview again:")
    vals, _ = _rows(d, T, 1)
    _same(live.push(**vals), _full(d, T + 1, prm), T, "committed after the preview:")
    vals, _ = _rows(d, T + 1, 5)
    _same(live.push(**vals), _full(d, T + 6, prm), T + 1, "next push:")
    live.close()


def test_multi_wave_panel_filled_on_the_device():
    """20,000 random-walk symbols (625 warps); the history is generated on the device and never crosses PCIe.  Candle rows
    only look back, so the rows of one recompute over all T + 73 bars are the recompute's rows at every push (and the
    last push's recompute is that panel exactly)."""
    S, T, pushes = 20000, 300, (1, 8, 64)
    n = T + sum(pushes)
    big = candles.CandlePanel(S, n)
    big.fill_random_walk(seed=77, sigma=0.02, to_host=True)
    big.run_host()
    d = {f: np.ascontiguousarray(big.host_field(i)) for i, f in enumerate(F4)}
    names = candles.pattern_names()
    full = ({names[k]: big.pattern(k).copy() for k in range(N.N_PATTERNS)},
            {N.PRICE_NAMES[q]: tuple(x.copy() for x in big.price(q)) for q in range(N.N_PRICES)})
    big.close()
    hist = candles.CandlePanel(S, T)
    hist.fill_random_walk(seed=77, sigma=0.02, to_host=False)
    live = hist.live(max_push_bars=64)
    hist.close()
    t = T
    for k in pushes:
        vals, _ = _rows(d, t, k)
        assert _same(live.push(**vals), full, t, f"push of {k} at bar {t}:") > 0
        t += k
    assert live.bars == n
    live.close()


def test_against_the_oracle(g):
    from oracle import pqo
    d, T, K = _golden(g), 200, 40
    hist = _panel(d, T, _params())
    hist.run_host()
    live = hist.live(max_push_bars=K)
    hist.close()
    vals, _ = _rows(d, T, K)
    pats, prices = live.push(**vals)
    names = candles.pattern_names()
    for s in (0, 13, 49):
        o, h, l, c = (d[f][s, :T + K] for f in F4)
        for k, name in enumerate(names):
            assert np.array_equal(pats[name][s], pqo.cdl(k, o, h, l, c)[T:]), (name, s)
        for q, name in enumerate(N.PRICE_NAMES):
            assert np.array_equal(prices[name][0][s].view(np.uint64), pqo.price(q, o, h, l, c)[T:].view(np.uint64)), (name, s)
    live.close()
