"""Null-aware live panels without a GPU: the C ABI answers PQB_ERR_NO_DEVICE, LivePanel checks `nulls=` / `valid=` before
anything reaches the native library, and the header documents the flag and the outputs a new null can void."""
import ctypes as C
import re
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parents[1]


@pytest.fixture(scope="module")
def N():
    from polars_quant_b200 import _native as N
    N.build()
    return N


def test_create_ex_without_a_device_is_no_device(N):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    out = C.c_void_p()
    for flags in (0, N.LIVE_NULLS):
        rc = N.lib().pqb_live_create_ex(None, C.byref(N.default_params()), 0, 64, flags, C.byref(out))
        assert rc == -1 and not out.value                 # PQB_ERR_NO_DEVICE
        assert b"no CPU fallback" in N.lib().pqb_last_error()
    assert not N.lib().pqb_live_host_voided(None, N.OUTPUT_NAMES.index("macd"))


def test_nulls_must_be_a_bool(N):
    from polars_quant_b200.live import LivePanel

    class Shell:                                           # (the check comes before any use of the panel)
        n_symbols = 5

    for bad in ("yes", 1, None):
        with pytest.raises(TypeError):
            LivePanel(Shell(), nulls=bad)


def _unbound(n_symbols=5, max_push=4):
    from polars_quant_b200.live import LivePanel
    lp = LivePanel.__new__(LivePanel)
    lp.n_symbols, lp.max_push_bars, lp._h, lp.outputs, lp.nulls = n_symbols, max_push, None, [], True
    return lp


@pytest.mark.parametrize("valid", [
    np.ones((2, 6), dtype=bool),                                          # wrong symbol count
    {"close": np.ones((3, 5), dtype=bool)},                               # wrong bar count
    {"open": np.ones((2, 5), dtype=bool)},                                # not a suite field
    {"close": np.ones((1, 2, 5), dtype=bool)},                            # three dimensions
])
def test_valid_shape_errors_on_a_null_aware_panel(N, valid):
    with pytest.raises(ValueError):
        _unbound().push(np.zeros((2, 5)), np.zeros((2, 5)), np.zeros((2, 5)), np.zeros((2, 5)), valid=valid)


def test_a_strict_panel_reports_no_voided_columns(N):
    from polars_quant_b200.live import LivePanel
    assert LivePanel.voided == {} and LivePanel.nulls is False


def test_header_documents_the_flag_and_the_voidable_outputs():
    h = (ROOT / "include" / "pqb200.h").read_text()
    assert re.search(r"enum \{ PQB_LIVE_NULLS = 1 \};", h)
    assert "pqb_live_create_ex(" in h and "pqb_live_host_voided(" in h
    doc = h[h.index("Null-aware live panels"):h.index("PQB_LIVE_NULLS = 1")]
    rules = {"close:": ["macd", "macd_signal", "macd_hist", "rsi"], "close, high or low:": ["willr"],
             "high or low:": ["midprice", "donchian_upper", "donchian_lower"]}
    for field, outs in rules.items():
        line = next(ln for ln in doc.splitlines() if ln.strip(" *").startswith(field))
        for o in outs:
            assert re.search(r"\b%s\b" % o, line), (field, o)
