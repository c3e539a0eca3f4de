"""Live panels without a GPU: the C ABI refuses to create one (no CPU fallback), and LivePanel.push checks shapes and
dtypes on the host before anything reaches the native library."""
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
    out = C.c_void_p()
    rc = N.lib().pqb_live_create(None, C.byref(N.default_params()), 0, 64, C.byref(out))
    assert rc == -1 and not out.value                     # PQB_ERR_NO_DEVICE
    assert b"no CPU fallback" in N.lib().pqb_last_error()
    assert N.lib().pqb_live_bars(None) == 0 and N.lib().pqb_live_state_bytes(None) == 0
    assert N.lib().pqb_live_push(None, 1, *([None] * 8), 1) == -3  # PQB_ERR_INVALID
    assert not N.lib().pqb_live_host_output(None, 0) and not N.lib().pqb_live_host_validity(None, 0)


def _unbound(n_symbols=5, max_push=4):
    """A LivePanel shell without a native object: push() must refuse its arguments before it calls the library."""
    from polars_quant_b200.live import LivePanel
    lp = LivePanel.__new__(LivePanel)
    lp.n_symbols, lp.max_push_bars, lp._h, lp.outputs = n_symbols, max_push, None, []
    return lp


@pytest.mark.parametrize("bad", [
    dict(close=np.zeros((2, 6))),                                        # wrong symbol count
    dict(close=np.zeros(4)),                                             # one bar, wrong symbol count
    dict(close=np.zeros((1, 2, 5))),                                     # three dimensions
    dict(close=np.zeros((2, 5)), high=np.zeros((3, 5))),                 # fields with different bar counts
    dict(close=np.zeros((5, 5))),                                        # more bars than max_push_bars
    dict(close=np.zeros((2, 5)), valid=np.ones((2, 4), dtype=bool)),     # validity of the wrong shape
    dict(close=np.zeros((2, 5)), valid={"open": np.ones((2, 5), dtype=bool)}),   # not a suite field
])
def test_push_shape_errors(N, bad):
    with pytest.raises(ValueError):
        _unbound().push(**bad)


def test_push_dtype_errors(N):
    with pytest.raises(ValueError):
        _unbound().push(np.array([["a"] * 5]))
    with pytest.raises(TypeError):
        _unbound().push({"close": np.zeros(5)})
