"""ctypes binding of libpqb200.so (include/pqb200.h).  There is no fallback: if the shared
library is missing, or no B200 is present when a compute entry point is called, this raises."""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from pathlib import Path

_PKG = Path(__file__).resolve().parent
LIB_PATH = Path(os.environ["PQB_LIB"]) if os.environ.get("PQB_LIB") else _PKG / "libpqb200.so"

N_FIELDS = 4
N_OUTPUTS = 44
N_SUITE_OUTPUTS = 21      # the 15-indicator benchmark suite; 21.. = optional groups
CLOSE, HIGH, LOW, VOLUME = 0, 1, 2, 3
OUTPUT_NAMES = ["sma", "ema", "tema", "trima", "bb_upper", "bb_middle", "bb_lower", "macd",
                "macd_signal", "macd_hist", "rsi", "trange", "atr", "natr", "obv", "ad",
                "kdj_k", "kdj_d", "kdj_j", "willr", "midprice",
                "midpoint", "adosc", "mom", "roc", "rocp", "rocr", "rocr100", "cmo", "mfi", "cci",
                "plus_dm", "minus_dm", "dx", "minus_di", "adx", "adxr", "trix", "ultosc", "aroon_up", "aroon_down",
                "donchian_upper", "donchian_lower", "fastk"]
IND = {"sma": 1 << 0, "ema": 1 << 1, "tema": 1 << 2, "trima": 1 << 3, "bbands": 1 << 4, "macd": 1 << 5,
       "rsi": 1 << 6, "trange": 1 << 7, "atr": 1 << 8, "natr": 1 << 9, "obv": 1 << 10, "ad": 1 << 11,
       "kdj": 1 << 12, "willr": 1 << 13, "midprice": 1 << 14}
IND_EXTRA = {"midpoint": 1 << 15, "adosc": 1 << 16, "mom": 1 << 17, "roc": 1 << 18, "cmo": 1 << 19, "mfi": 1 << 20,
             "cci": 1 << 21, "dm": 1 << 22, "trix": 1 << 23, "ultosc": 1 << 24, "aroon": 1 << 25,
             "donchian": 1 << 26}
IND_ALL = (1 << 15) - 1
IND_FASTK = 1 << 27          # with IND["kdj"]: also store the raw %K line (output "fastk"); opt-in, the general kernel only
LIVE_NULLS = 1               # pqb_live_create_ex flag: null-aware live panel (include/pqb200.h)

ERR_NAMES = {-1: "PQB_ERR_NO_DEVICE", -2: "PQB_ERR_CUDA", -3: "PQB_ERR_INVALID", -4: "PQB_ERR_UNSUPPORTED",
             -5: "PQB_ERR_NULLS", -6: "PQB_ERR_ALLOC"}


class PqbError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__("%s: %s" % (ERR_NAMES.get(code, code), msg))
        self.code = code


class SuiteParams(C.Structure):
    _fields_ = [("indicators", C.c_uint32), ("sma_period", C.c_int32), ("ema_period", C.c_int32),
                ("tema_period", C.c_int32), ("trima_period", C.c_int32), ("bbands_period", C.c_int32),
                ("bbands_nbdevup", C.c_double), ("bbands_nbdevdn", C.c_double), ("macd_fast", C.c_int32),
                ("macd_slow", C.c_int32), ("macd_signal", C.c_int32), ("rsi_period", C.c_int32),
                ("atr_period", C.c_int32), ("natr_period", C.c_int32), ("kdj_fastk", C.c_int32),
                ("kdj_slowk", C.c_int32), ("kdj_slowd", C.c_int32), ("willr_period", C.c_int32),
                ("midprice_period", C.c_int32), ("midpoint_period", C.c_int32), ("adosc_fast", C.c_int32),
                ("adosc_slow", C.c_int32), ("mom_period", C.c_int32), ("roc_period", C.c_int32),
                ("cmo_period", C.c_int32), ("mfi_period", C.c_int32), ("cci_period", C.c_int32), ("dm_period", C.c_int32),
                ("trix_period", C.c_int32), ("ultosc_period1", C.c_int32), ("ultosc_period2", C.c_int32),
                ("ultosc_period3", C.c_int32), ("aroon_period", C.c_int32), ("donchian_period", C.c_int32)]


class CandleParams(C.Structure):
    _fields_ = [("patterns", C.c_uint64), ("prices", C.c_uint32), ("pen_darkcloudcover", C.c_double),
                ("pen_eveningdojistar", C.c_double), ("pen_eveningstar", C.c_double),
                ("pen_morningdojistar", C.c_double), ("pen_morningstar", C.c_double), ("pen_piercing", C.c_double)]


class LiveScreen(C.Structure):
    """pqb_live_screen: what a live panel's screen serves (include/pqb200.h "live screens")."""
    _fields_ = [("oversold", C.c_double), ("overbought", C.c_double), ("ma_type", C.c_int32), ("ma_fast", C.c_int32),
                ("ma_slow", C.c_int32), ("info", C.c_int32)]


N_PATTERNS = 61
N_PRICES = 5
PRICE_NAMES = ["avgprice", "medprice", "typprice", "wclprice", "bop"]
INFO_NAMES = ["price", "high", "low", "volume", "return_1d", "return_5d", "return_20d", "volatility", "ma_5", "ma_10",
              "ma_20", "volume_ratio", "amplitude"]      # enum pqb_info
OPEN_, HIGH_, LOW_, CLOSE_ = 0, 1, 2, 3          # candle panel fields


class Col(C.Structure):
    _fields_ = [("values", C.c_void_p), ("validity", C.c_void_p), ("offset", C.c_int64), ("len", C.c_int64)]


class ColRef(C.Structure):
    """pqb_col_ref: one caller-owned Arrow f64 column and the (symbol, field) it goes to."""
    _fields_ = [("values", C.c_void_p), ("validity", C.c_void_p), ("offset", C.c_int64), ("len", C.c_int64),
                ("symbol", C.c_int64), ("field", C.c_int32), ("reserved", C.c_int32)]


class ArrowSchema(C.Structure):
    pass


class ArrowArray(C.Structure):
    pass


ArrowSchema._fields_ = [("format", C.c_char_p), ("name", C.c_char_p), ("metadata", C.c_char_p), ("flags", C.c_int64),
                        ("n_children", C.c_int64), ("children", C.POINTER(C.POINTER(ArrowSchema))),
                        ("dictionary", C.POINTER(ArrowSchema)), ("release", C.c_void_p), ("private_data", C.c_void_p)]
ArrowArray._fields_ = [("length", C.c_int64), ("null_count", C.c_int64), ("offset", C.c_int64), ("n_buffers", C.c_int64),
                       ("n_children", C.c_int64), ("buffers", C.POINTER(C.c_void_p)),
                       ("children", C.POINTER(C.POINTER(ArrowArray))), ("dictionary", C.POINTER(ArrowArray)),
                       ("release", C.c_void_p), ("private_data", C.c_void_p)]


class OutCol(C.Structure):
    _fields_ = [("values", C.c_void_p), ("validity", C.c_void_p)]


def build(force: bool = False) -> Path:
    """Compiles libpqb200.so in-tree with nvcc for sm_100a (works without a GPU)."""
    srcs = (list((_PKG / "csrc").glob("*.cu*")) + list((_PKG / "csrc").glob("*.inc")) +
            list((_PKG.parent / "include").glob("*.h")))
    if force or not LIB_PATH.exists() or any(s.stat().st_mtime > LIB_PATH.stat().st_mtime for s in srcs):
        r = subprocess.run(["make", "-C", str(_PKG / "csrc"), "-B"], capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("building libpqb200.so failed:\n" + r.stdout + r.stderr)
    return LIB_PATH


_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        if not LIB_PATH.exists():
            raise RuntimeError("libpqb200.so is not built (run python -c 'import __graft_entry__ as g; g.build()'); "
                               "there is no CPU fallback")
        L = C.CDLL(str(LIB_PATH))
        L.pqb_last_error.restype = C.c_char_p
        L.pqb_panel_pitch.restype = C.c_int64
        L.pqb_panel_pitch.argtypes = [C.c_void_p]
        L.pqb_panel_validity_pitch.restype = C.c_int64
        L.pqb_panel_validity_pitch.argtypes = [C.c_void_p]
        for name in ("pqb_panel_host_field", "pqb_panel_host_output", "pqb_panel_host_validity",
                     "pqb_panel_device_field", "pqb_panel_device_output", "pqb_panel_device_validity"):
            f = getattr(L, name)
            f.restype = C.c_void_p
            f.argtypes = [C.c_void_p, C.c_int]
        L.pqb_engine_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
        L.pqb_engine_destroy.argtypes = [C.c_void_p]
        L.pqb_engine_destroy.restype = None
        L.pqb_panel_create.argtypes = [C.c_void_p, C.c_int64, C.c_int64, C.c_uint32, C.c_uint64, C.c_int,
                                       C.POINTER(C.c_void_p)]
        L.pqb_panel_destroy.argtypes = [C.c_void_p]
        L.pqb_panel_destroy.restype = None
        L.pqb_panel_set_column.argtypes = [C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64]
        L.pqb_panel_set_starts.argtypes = [C.c_void_p, C.c_void_p]
        L.pqb_panel_upload.argtypes = [C.c_void_p]
        L.pqb_panel_download.argtypes = [C.c_void_p]
        L.pqb_panel_sync.argtypes = [C.c_void_p]
        L.pqb_suite_run.argtypes = [C.c_void_p, C.POINTER(SuiteParams)]
        L.pqb_suite_run_host.argtypes = [C.c_void_p, C.POINTER(SuiteParams), C.c_int64]
        L.pqb_panel_set_columns.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int]
        L.pqb_suite_run_columns.argtypes = [C.c_void_p, C.POINTER(SuiteParams), C.c_void_p, C.c_int64, C.c_int]
        L.pqb_panel_set_record_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
        L.pqb_suite_run_record_batch.argtypes = [C.c_void_p, C.POINTER(SuiteParams), C.c_void_p, C.c_void_p, C.c_void_p,
                                                 C.c_void_p, C.c_int]
        L.pqb_panel_export_arrow.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p]
        L.pqb_output_name.argtypes = [C.c_int]
        L.pqb_output_name.restype = C.c_char_p
        L.pqb_engine_local_cpus.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
        L.pqb_panel_get_output.argtypes = [C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_void_p, C.c_int64]
        L.pqb_panel_fill_synthetic.argtypes = [C.c_void_p, C.c_uint64, C.c_double, C.c_int]
        L.pqb_suite_time.argtypes = [C.c_void_p, C.POINTER(SuiteParams), C.c_int, C.c_int, C.POINTER(C.c_float),
                                     C.POINTER(C.c_float), C.POINTER(C.c_int)]
        L.pqb_suite_time_host.argtypes = [C.c_void_p, C.POINTER(SuiteParams), C.c_int64, C.c_int, C.c_int,
                                          C.POINTER(C.c_float)]
        L.pqb_flush_l2.argtypes = [C.c_void_p]
        L.pqb_stream_mix.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int64, C.c_int, C.c_int, C.POINTER(C.c_float)]
        L.pqb_probe_pcie.argtypes = [C.c_void_p, C.c_int64, C.c_int, C.POINTER(C.c_double)]
        L.pqb_panel_clear_validity.argtypes = [C.c_void_p, C.c_int]
        L.pqb_donchian.argtypes = [C.c_void_p, C.POINTER(Col), C.POINTER(Col), C.c_int32, C.POINTER(OutCol), C.POINTER(OutCol)]
        L.pqb_dm.argtypes = [C.c_void_p, C.POINTER(Col), C.POINTER(Col), C.POINTER(Col), C.c_int32] + [C.POINTER(OutCol)] * 6
        L.pqb_selftest_divsqrt.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(C.c_uint64)]
        L.pqb_multi_destroy.argtypes = [C.c_void_p]
        L.pqb_multi_destroy.restype = None
        L.pqb_multi_shard_count.argtypes = [C.c_void_p]
        L.pqb_multi_run_host.argtypes = [C.c_void_p, C.POINTER(SuiteParams)]
        L.pqb_panel_last_launches.argtypes = [C.c_void_p]
        L.pqb_panel_tiled_shape.argtypes = [C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
        L.pqb_suite_params_default.argtypes = [C.POINTER(SuiteParams)]
        L.pqb_suite_params_default.restype = None
        L.pqb_signals_run.argtypes = [C.c_void_p, C.c_double, C.c_double]
        L.pqb_ma_cross_run.argtypes = [C.c_void_p, C.c_int, C.c_int32, C.c_int32]
        L.pqb_panel_host_signal.argtypes = [C.c_void_p, C.c_int]
        L.pqb_panel_host_signal.restype = C.c_void_p
        L.pqb_panel_device_signal.argtypes = [C.c_void_p, C.c_int]
        L.pqb_panel_device_signal.restype = C.c_void_p
        L.pqb_signals_time.argtypes = [C.c_void_p, C.c_double, C.c_double, C.c_int, C.c_int, C.POINTER(C.c_float)]
        L.pqb_panel_info.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        # time-split panels
        L.pqb_split_required_warmup.argtypes = [C.POINTER(SuiteParams)]
        L.pqb_split_required_warmup.restype = C.c_int64
        L.pqb_split_create.argtypes = [C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_uint32, C.c_uint64, C.c_int,
                                       C.POINTER(C.c_void_p)]
        L.pqb_split_destroy.argtypes = [C.c_void_p]
        L.pqb_split_destroy.restype = None
        L.pqb_split_panel.argtypes = [C.c_void_p]
        L.pqb_split_panel.restype = C.c_void_p
        L.pqb_split_shape.argtypes = [C.c_void_p] + [C.POINTER(C.c_int64)] * 4
        L.pqb_split_set_column.argtypes = [C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64]
        L.pqb_split_run.argtypes = [C.c_void_p, C.POINTER(SuiteParams)]
        L.pqb_split_run_host.argtypes = [C.c_void_p, C.POINTER(SuiteParams)]
        L.pqb_split_get_output.argtypes = [C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_void_p, C.c_int64]
        L.pqb_split_fill_synthetic.argtypes = [C.c_void_p, C.c_uint64, C.c_double]
        # long rows (config 3)
        L.pqb_long_create.argtypes = [C.c_void_p, C.c_int64, C.c_int64, C.c_int, C.c_int, C.c_int64, C.c_int, C.POINTER(C.c_void_p)]
        L.pqb_long_destroy.argtypes = [C.c_void_p]
        L.pqb_long_destroy.restype = None
        L.pqb_long_panel.argtypes = [C.c_void_p]
        L.pqb_long_panel.restype = C.c_void_p
        L.pqb_long_run.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int32, C.c_int32, C.c_int32]
        L.pqb_long_last_launches.argtypes = [C.c_void_p]
        L.pqb_long_time.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int32, C.c_int32, C.c_int32, C.c_int, C.c_int, C.POINTER(C.c_float)]
        # many windows in one launch (config 5)
        L.pqb_windows_create.argtypes = [C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_int, C.c_int32, C.c_int32, C.c_void_p,
                                         C.c_int, C.c_int32, C.c_int, C.POINTER(C.c_void_p)]
        L.pqb_windows_destroy.argtypes = [C.c_void_p]
        L.pqb_windows_destroy.restype = None
        L.pqb_windows_panel.argtypes = [C.c_void_p]
        L.pqb_windows_panel.restype = C.c_void_p
        L.pqb_windows_slot.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int]
        L.pqb_windows_run.argtypes = [C.c_void_p]
        L.pqb_windows_last_launches.argtypes = [C.c_void_p]
        L.pqb_windows_time.argtypes = [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_float)]
        L.pqb_windows_live_create.argtypes = [C.c_void_p, C.c_int64, C.POINTER(C.c_void_p)]
        L.pqb_windows_live_destroy.argtypes = [C.c_void_p]
        L.pqb_windows_live_destroy.restype = None
        L.pqb_windows_live_bars.argtypes = [C.c_void_p]
        L.pqb_windows_live_bars.restype = C.c_int64
        L.pqb_windows_live_state_bytes.argtypes = [C.c_void_p]
        L.pqb_windows_live_state_bytes.restype = C.c_int64
        L.pqb_windows_live_push.argtypes = [C.c_void_p, C.c_int64] + [C.c_void_p] * 6 + [C.c_int]
        for name in ("pqb_windows_live_host_output", "pqb_windows_live_host_validity", "pqb_windows_live_host_voided"):
            f = getattr(L, name)
            f.restype = C.c_void_p
            f.argtypes = [C.c_void_p, C.c_int]
        L.pqb_windows_live_last_push_ms.argtypes = [C.c_void_p, C.POINTER(C.c_float)]
        # candle engine
        L.pqb_candle_params_default.argtypes = [C.POINTER(CandleParams)]
        L.pqb_candle_params_default.restype = None
        L.pqb_pattern_name.argtypes = [C.c_int]
        L.pqb_pattern_name.restype = C.c_char_p
        L.pqb_pattern_index.argtypes = [C.c_char_p]
        L.pqb_candles_create.argtypes = [C.c_void_p, C.c_int64, C.c_int64, C.c_uint64, C.c_uint32, C.c_int,
                                         C.POINTER(C.c_void_p)]
        L.pqb_candles_destroy.argtypes = [C.c_void_p]
        L.pqb_candles_destroy.restype = None
        L.pqb_candles_pitch.argtypes = [C.c_void_p]
        L.pqb_candles_pitch.restype = C.c_int64
        L.pqb_candles_set_column.argtypes = [C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64]
        for name in ("pqb_candles_host_field", "pqb_candles_host_pattern", "pqb_candles_host_price",
                     "pqb_candles_host_price_validity"):
            f = getattr(L, name)
            f.restype = C.c_void_p
            f.argtypes = [C.c_void_p, C.c_int]
        L.pqb_candles_run.argtypes = [C.c_void_p, C.POINTER(CandleParams)]
        L.pqb_candles_run_host.argtypes = [C.c_void_p, C.POINTER(CandleParams)]
        L.pqb_candles_get_pattern.argtypes = [C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_int64]
        L.pqb_candles_get_price.argtypes = [C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_void_p, C.c_int64]
        L.pqb_candles_fill_synthetic.argtypes = [C.c_void_p, C.c_uint64, C.c_int]
        L.pqb_candles_fill_random_walk.argtypes = [C.c_void_p, C.c_uint64, C.c_double, C.c_int]
        L.pqb_candles_time.argtypes = [C.c_void_p, C.POINTER(CandleParams), C.c_int, C.c_int, C.POINTER(C.c_float)]
        L.pqb_cdl.argtypes = [C.c_void_p, C.c_int, C.POINTER(Col), C.POINTER(Col), C.POINTER(Col), C.POINTER(Col),
                              C.c_double, C.c_void_p]
        L.pqb_price.argtypes = [C.c_void_p, C.c_int, C.POINTER(Col), C.POINTER(Col), C.POINTER(Col), C.POINTER(Col),
                                C.POINTER(OutCol)]
        # live candle panels
        L.pqb_candles_live_create.argtypes = [C.c_void_p, C.POINTER(CandleParams), C.c_int64, C.POINTER(C.c_void_p)]
        L.pqb_candles_live_destroy.argtypes = [C.c_void_p]
        L.pqb_candles_live_destroy.restype = None
        L.pqb_candles_live_bars.argtypes = [C.c_void_p]
        L.pqb_candles_live_bars.restype = C.c_int64
        L.pqb_candles_live_push.argtypes = [C.c_void_p, C.c_int64] + [C.c_void_p] * 8 + [C.c_int]
        for name in ("pqb_candles_live_host_pattern", "pqb_candles_live_host_price", "pqb_candles_live_host_price_validity"):
            f = getattr(L, name)
            f.restype = C.c_void_p
            f.argtypes = [C.c_void_p, C.c_int]
        L.pqb_candles_live_last_push_ms.argtypes = [C.c_void_p, C.POINTER(C.c_float)]
        # live panels
        L.pqb_live_create.argtypes = [C.c_void_p, C.POINTER(SuiteParams), C.c_uint64, C.c_int64, C.POINTER(C.c_void_p)]
        L.pqb_live_destroy.argtypes = [C.c_void_p]
        L.pqb_live_destroy.restype = None
        L.pqb_live_bars.argtypes = [C.c_void_p]
        L.pqb_live_bars.restype = C.c_int64
        L.pqb_live_state_bytes.argtypes = [C.c_void_p]
        L.pqb_live_state_bytes.restype = C.c_int64
        L.pqb_live_push.argtypes = [C.c_void_p, C.c_int64] + [C.c_void_p] * 8 + [C.c_int]
        L.pqb_live_host_output.argtypes = [C.c_void_p, C.c_int]
        L.pqb_live_host_output.restype = C.c_void_p
        L.pqb_live_host_validity.argtypes = [C.c_void_p, C.c_int]
        L.pqb_live_host_validity.restype = C.c_void_p
        L.pqb_live_last_push_ms.argtypes = [C.c_void_p, C.POINTER(C.c_float)]
        L.pqb_live_create_ex.argtypes = [C.c_void_p, C.POINTER(SuiteParams), C.c_uint64, C.c_int64, C.c_uint32,
                                         C.POINTER(C.c_void_p)]
        L.pqb_live_host_voided.argtypes = [C.c_void_p, C.c_int]
        L.pqb_live_host_voided.restype = C.c_void_p
        L.pqb_live_screen_default.argtypes = [C.POINTER(LiveScreen)]
        L.pqb_live_screen_default.restype = None
        L.pqb_live_create_screen.argtypes = [C.c_void_p, C.POINTER(SuiteParams), C.c_uint64, C.c_int64, C.c_uint32,
                                             C.POINTER(LiveScreen), C.POINTER(C.c_void_p)]
        L.pqb_live_host_signal.argtypes = [C.c_void_p, C.c_int]
        L.pqb_live_host_signal.restype = C.c_void_p
        L.pqb_live_host_info.argtypes = [C.c_void_p]
        L.pqb_live_host_info.restype = C.c_void_p
        L.pqb_live_host_info_valid.argtypes = [C.c_void_p]
        L.pqb_live_host_info_valid.restype = C.c_void_p
        L.pqb_live_info.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        _lib = L
    return _lib


def check(rc: int):
    if rc != 0:
        raise PqbError(rc, lib().pqb_last_error().decode("utf-8", "replace"))


def default_params(indicators: int = IND_ALL, **overrides) -> SuiteParams:
    p = SuiteParams()
    lib().pqb_suite_params_default(C.byref(p))
    p.indicators = indicators
    for k, v in overrides.items():
        if not hasattr(p, k):
            raise TypeError("unknown suite parameter %r" % k)
        setattr(p, k, v)
    return p
