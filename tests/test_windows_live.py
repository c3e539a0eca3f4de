"""Live window panels without a GPU: the C ABI refuses to create one (no CPU fallback), and WindowLive.push checks shapes,
dtypes and fields on the host before anything reaches the native library."""
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
    assert L.pqb_windows_live_create(None, 64, C.byref(out)) == -1 and not out.value      # PQB_ERR_NO_DEVICE
    assert b"no CPU fallback" in L.pqb_last_error()
    assert L.pqb_windows_live_bars(None) == 0 and L.pqb_windows_live_state_bytes(None) == 0
    assert L.pqb_windows_live_push(None, 1, *([None] * 6), 1) == -3                        # PQB_ERR_INVALID
    for name in ("pqb_windows_live_host_output", "pqb_windows_live_host_validity", "pqb_windows_live_host_voided"):
        assert not getattr(L, name)(None, 0)
    ms = C.c_float()
    assert L.pqb_windows_live_last_push_ms(None, C.byref(ms)) == -3
    L.pqb_windows_live_destroy(None)


def _unbound(n_symbols=5, max_push=4):
    """A WindowLive shell without a native object: push() must refuse its arguments before it calls the library."""
    from polars_quant_b200.windows import WindowLive
    wl = WindowLive.__new__(WindowLive)
    wl.n_symbols, wl.max_push_bars, wl._h, wl.names = n_symbols, max_push, None, {}
    return wl


Z = np.zeros((2, 5))


@pytest.mark.parametrize("bad", [
    dict(close=np.zeros((2, 6)), high=np.zeros((2, 6)), low=np.zeros((2, 6))),      # wrong symbol count
    dict(close=np.zeros(4), high=np.zeros(4), low=np.zeros(4)),                      # one bar, wrong symbol count
    dict(close=np.zeros((1, 2, 5)), high=Z, low=Z),                                  # three dimensions
    dict(close=Z, high=np.zeros((3, 5)), low=Z),                                     # fields with different bar counts
    dict(close=Z, high=Z, low=None),                                                 # a missing field
    dict(close=np.zeros((5, 5)), high=np.zeros((5, 5)), low=np.zeros((5, 5))),       # more bars than max_push_bars
    dict(close=Z, high=Z, low=Z, valid=np.ones((2, 4), dtype=bool)),                 # validity of the wrong shape
    dict(close=Z, high=Z, low=Z, valid={"volume": np.ones((2, 5), dtype=bool)}),    # not a field of a window panel
])
def test_push_argument_errors(N, bad):
    with pytest.raises(ValueError):
        _unbound().push(**bad)


def test_push_dtype_errors(N):
    with pytest.raises(ValueError):
        _unbound().push(np.array([["a"] * 5]), Z[:1], Z[:1])
    with pytest.raises(TypeError):
        _unbound().push({"close": np.zeros(5)}, Z[:1], Z[:1])


def test_header_documents_the_section():
    from pathlib import Path
    h = (Path(__file__).resolve().parents[1] / "include" / "pqb200.h").read_text()
    i = h.index("live window panels")
    assert h.index("many rolling windows") < i
    sec = h[i:h.index("pqb_windows_live_last_push_ms")]
    for word in ("willr", "midprice", "donchian_upper", "preview", "PQB_ERR_UNSUPPORTED", "one host thread per engine"):
        assert word in sec, word
