"""Time-split panels (BASELINE config 3: few symbols, very long rows): each row runs as `chunks` independent
virtual symbols with a warm-up of real history.  Chunk 0 is the reference's computation bit for bit; later chunks
must agree with the serial oracle within the north-star tolerance (rel 1e-10 / abs 1e-12); pure window functions
and validity must be exact."""
import numpy as np
import pytest

import synth
import tolerances as T
from oracle import pqo
from polars_quant_b200 import _native as N

pytestmark = pytest.mark.gpu
REL, ABS = 1e-10, 1e-12


@pytest.fixture(scope="module")
def pq():
    import polars_quant_b200 as pq
    return pq


def _close_enough(name, got, ref):
    (gv, gok), (rv, rok) = got, ref
    assert np.array_equal(gok, rok), f"{name}: validity differs"
    d = np.abs(gv[rok] - rv[rok])
    lim = ABS + REL * np.abs(rv[rok])
    assert (d <= lim).all(), f"{name}: max err {d.max():.3e} (worst rel {(d / np.maximum(np.abs(rv[rok]), 1e-300)).max():.3e})"
    return float(T.same_bits(gv[rok], rv[rok]).mean())


def test_config3_ema_macd_split_against_the_serial_oracle(pq):
    S, NB = 5, 400_000
    d = synth.ohlcv(S, NB, seed=3, sigma=0.0005)
    om = sum(1 << pqo.OUTPUT_NAMES.index(o) for o in ("ema", "macd", "macd_signal", "macd_hist"))
    for period, chunks in ((12, 16), (200, 16), (5000, 4)):
        prm = N.default_params(indicators=N.IND["ema"] | N.IND["macd"], ema_period=period)
        W = pq.SplitPanel.required_warmup(prm)
        p = pq.SplitPanel(S, NB, chunks=chunks, warmup=W, fields_mask=1, outputs_mask=om)
        assert p.virtual_symbols == S * chunks and p.warmup >= W
        p.set_fields(close=d["close"])
        p.run_host(prm)
        for s in range(S):
            exact = _close_enough(f"ema({period})", p.get_output(s, pqo.OUTPUT_NAMES.index("ema")), pqo.ema(d["close"][s], period))
            assert exact > 0.9                        # the warm-up mostly converges to the serial trajectory's own bits
            for name, ref in zip(("macd", "macd_signal", "macd_hist"), pqo.macd(d["close"][s], 12, 26, 9)):
                _close_enough(name, p.get_output(s, pqo.OUTPUT_NAMES.index(name)), ref)
            # chunk 0 is the reference's computation itself
            v, ok = p.get_output(s, pqo.OUTPUT_NAMES.index("ema"))
            rv, rok = pqo.ema(d["close"][s], period)
            assert T.same_bits(v[:p.chunk_bars][rok[:p.chunk_bars]], rv[:p.chunk_bars][rok[:p.chunk_bars]]).all()
        p.close()


def test_ema_and_macd_at_a_high_price_level(pq):
    """Price level 1e5, where one ulp of the price (1.5e-11) is larger than abs 1e-12: a chunk's warm-up converges to the
    serial state's own bits, so the MACD lines, which cross zero, still meet rel 1e-10 / abs 1e-12 (measured on a B200:
    the MACD lines bit-identical to the serial oracle)."""
    S, NB, period = 5, 400_000, 12
    close = synth.ohlcv(S, NB, seed=3, sigma=0.0005)["close"] * 1e3
    om = sum(1 << pqo.OUTPUT_NAMES.index(o) for o in ("ema", "macd", "macd_signal", "macd_hist"))
    prm = N.default_params(indicators=N.IND["ema"] | N.IND["macd"], ema_period=period)
    p = pq.SplitPanel(S, NB, chunks=16, warmup=pq.SplitPanel.required_warmup(prm), fields_mask=1, outputs_mask=om)
    p.set_fields(close=close)
    p.run_host(prm)
    for s in range(S):
        _close_enough("ema", p.get_output(s, pqo.OUTPUT_NAMES.index("ema")), pqo.ema(close[s], period))
        for name, ref in zip(("macd", "macd_signal", "macd_hist"), pqo.macd(close[s], 12, 26, 9)):
            _close_enough(name, p.get_output(s, pqo.OUTPUT_NAMES.index(name)), ref)
    p.close()


def test_split_suite_recurrences_and_window_functions(pq):
    S, NB = 4, 60_000
    d = synth.ohlcv(S, NB, seed=8)
    names = ("ema", "tema", "macd", "macd_signal", "macd_hist", "rsi", "trange", "atr", "natr", "willr", "midprice")
    ind = sum(N.IND[k] for k in ("ema", "tema", "macd", "rsi", "trange", "atr", "natr", "willr", "midprice"))
    for k in ("sma", "trima", "bbands", "kdj", "obv", "ad"):          # running sums / cumulative: history-dependent
        assert pq.SplitPanel.required_warmup(N.default_params(indicators=N.IND[k])) == -1, k
    prm = N.default_params(indicators=ind)
    om = sum(1 << pqo.OUTPUT_NAMES.index(o) for o in names)
    p = pq.SplitPanel(S, NB, chunks=8, warmup=pq.SplitPanel.required_warmup(prm), outputs_mask=om)
    p.set_fields(d["close"], d["high"], d["low"], d["volume"])
    p.run_host(prm)
    out, ok, _ = pqo.suite_panel(d["close"], d["high"], d["low"], d["volume"])
    for s in range(S):
        for n in names:
            k = pqo.OUTPUT_NAMES.index(n)
            exact = _close_enough(n, p.get_output(s, k), (out[k][s], ok[k][s]))
            if n in ("trange", "willr", "midprice"):
                assert exact == 1.0, n                 # pure window functions: bit-exact in every chunk
    p.close()


def test_split_refuses_what_cannot_be_split(pq):
    prm = N.default_params()                           # the full suite contains OBV and AD
    assert pq.SplitPanel.required_warmup(prm) == -1
    p = pq.SplitPanel(2, 4096, chunks=4, warmup=64)
    x = np.linspace(1.0, 2.0, 4096)
    for f in range(4):
        p.set_column(0, f, x); p.set_column(1, f, x)
    with pytest.raises(N.PqbError) as e:
        p.run_host(prm)
    assert e.value.code == -4
    with pytest.raises(N.PqbError, match="warm-up"):
        p.run_host(N.default_params(indicators=N.IND["ema"], ema_period=30))      # needs 464 bars, has 64
    p.run_host(N.default_params(indicators=N.IND["willr"], willr_period=30))      # a 30-bar window fits
    v, ok = p.get_output(0, pqo.OUTPUT_NAMES.index("willr"))
    rv, rok = pqo.willr(x, x, x, 30)
    assert np.array_equal(ok, rok) and T.same_bits(v[ok], rv[rok]).all()
    p.close()
