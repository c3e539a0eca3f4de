"""Live candle panels without a GPU: the C ABI refuses to create one (no CPU fallback), and CandleLive.push checks shapes,
dtypes, fields and the push length on the host before anything reaches the native library."""
import ctypes as C

import numpy as np
import pytest


@pytest.fixture(scope="module")
def N():
    from polars_quant_b200 import _native as N
    N.build()
    return N


def test_create_without_a_device_is_no_device(N):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    L = N.lib()
    out = C.c_void_p()
    p = N.CandleParams()
    L.pqb_candle_params_default(C.byref(p))
    assert L.pqb_candles_live_create(None, C.byref(p), 64, C.byref(out)) == -1 and not out.value     # PQB_ERR_NO_DEVICE
    assert b"no CPU fallback" in L.pqb_last_error()
    assert L.pqb_candles_live_bars(None) == 0
    assert L.pqb_candles_live_push(None, 1, *([None] * 8), 1) == -3                                 # PQB_ERR_INVALID
    for name in ("pqb_candles_live_host_pattern", "pqb_candles_live_host_price", "pqb_candles_live_host_price_validity"):
        assert not getattr(L, name)(None, 0)
    ms = C.c_float()
    assert L.pqb_candles_live_last_push_ms(None, C.byref(ms)) == -3
    L.pqb_candles_live_destroy(None)


def _unbound(n_symbols=5, max_push=4):
    """A CandleLive shell without a native object: push() must refuse its arguments before it calls the library."""
    from polars_quant_b200.candles import CandleLive
    cl = CandleLive.__new__(CandleLive)
    cl.n_symbols, cl.max_push_bars, cl._h, cl.patterns, cl.prices = n_symbols, max_push, None, [], []
    return cl


Z = np.zeros((2, 5))


@pytest.mark.parametrize("bad", [
    dict(open=np.zeros((2, 6)), high=np.zeros((2, 6)), low=np.zeros((2, 6)), close=np.zeros((2, 6))),   # wrong symbol count
    dict(open=np.zeros(4), high=np.zeros(4), low=np.zeros(4), close=np.zeros(4)),                       # one bar, wrong count
    dict(open=np.zeros((1, 2, 5)), high=Z, low=Z, close=Z),                                             # three dimensions
    dict(open=Z, high=np.zeros((3, 5)), low=Z, close=Z),                                                # different bar counts
    dict(open=Z, high=Z, low=Z, close=np.zeros((1, 5))),
    dict(),                                                                                             # no field at all
    dict(open=np.zeros((5, 5)), high=np.zeros((5, 5)), low=np.zeros((5, 5)), close=np.zeros((5, 5))),   # k > max_push_bars
    dict(high=np.zeros((5, 5)), low=np.zeros((5, 5))),                                                  # ... prices only
    dict(open=Z, high=Z, low=Z, close=Z, valid=np.ones((2, 4), dtype=bool)),                            # validity shape
    dict(open=Z, high=Z, low=Z, close=Z, valid={"close": np.ones((3, 5), dtype=bool)}),                 # validity bar count
    dict(open=Z, high=Z, low=Z, close=Z, valid={"volume": np.ones((2, 5), dtype=bool)}),                # not a candle field
])
def test_push_argument_errors(N, bad):
    with pytest.raises(ValueError):
        _unbound().push(**bad)


def test_push_dtype_errors(N):
    with pytest.raises(ValueError):
        _unbound().push(np.array([["a"] * 5]), Z[:1], Z[:1], Z[:1])
    with pytest.raises(TypeError):
        _unbound().push({"open": np.zeros(5)}, Z[:1], Z[:1], Z[:1])


def test_header_documents_the_section():
    from pathlib import Path
    h = (Path(__file__).resolve().parents[1] / "include" / "pqb200.h").read_text()
    i = h.index("live candle panels")
    assert h.index("candle engine") < i
    sec = h[i:h.index("pqb_candles_live_last_push_ms")]
    for word in ("pqb_candles_live_create", "pqb_candles_live_push", "pqb_candles_live_host_pattern",
                 "pqb_candles_live_host_price_validity", "pqb_candles_live_bars", "pqb_candles_live_destroy",
                 "PQB_ERR_NULLS", "cont_slice", "avgprice", "medprice", "preview", "one host thread per engine",
                 "pqb_candles_fill_random_walk", "[k][n_symbols]"):
        assert word in sec, word
