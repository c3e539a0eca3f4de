"""Candle engine binding (include/pqb200.h "candle engine"): the reference's 61 cdl* patterns, the four
price transforms and BOP from one fused pass over an open / high / low / close panel."""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _native as N
from .panel import Engine, get_engine


def pattern_names() -> list[str]:
    return [N.lib().pqb_pattern_name(k).decode() for k in range(N.N_PATTERNS)]


def default_params(patterns: int | None = None, prices: int | None = None, penetration: float | None = None) -> N.CandleParams:
    p = N.CandleParams()
    N.lib().pqb_candle_params_default(C.byref(p))
    if patterns is not None:
        p.patterns = patterns
    if prices is not None:
        p.prices = prices
    if penetration is not None:
        for f in ("pen_darkcloudcover", "pen_eveningdojistar", "pen_eveningstar", "pen_morningdojistar",
                  "pen_morningstar", "pen_piercing"):
            setattr(p, f, float(penetration))
    return p


class CandlePanel:
    """open / high / low / close of `n_symbols` x `n_bars` on one B200 + the planes of the masked outputs."""

    def __init__(self, n_symbols: int, n_bars: int, engine: Engine | None = None, patterns_mask: int | None = None,
                 prices_mask: int | None = None, host_staging: bool = True):
        self.engine = engine or get_engine(0)
        self.n_symbols, self.n_bars = int(n_symbols), int(n_bars)
        self.patterns_mask = (1 << N.N_PATTERNS) - 1 if patterns_mask is None else int(patterns_mask)
        self.prices_mask = (1 << N.N_PRICES) - 1 if prices_mask is None else int(prices_mask)
        self._h = C.c_void_p()
        N.check(N.lib().pqb_candles_create(self.engine._h, self.n_symbols, self.n_bars, self.patterns_mask,
                                           self.prices_mask, 1 if host_staging else 0, C.byref(self._h)))
        self.pitch = N.lib().pqb_candles_pitch(self._h)
        self.words_per_row = (self.n_bars + 31) // 32

    def close(self):
        if self._h:
            N.lib().pqb_candles_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _view(self, ptr, dtype, cols):
        if not ptr:
            raise ValueError("this plane was not allocated")
        buf = (C.c_char * (self.n_symbols * cols * np.dtype(dtype).itemsize)).from_address(ptr)
        buf._owner = self                  # the view keeps the panel (and its pinned planes) alive, like Panel._view
        return np.frombuffer(buf, dtype=dtype).reshape(self.n_symbols, cols)

    def host_field(self, f: int) -> np.ndarray:
        return self._view(N.lib().pqb_candles_host_field(self._h, f), np.float64, self.pitch)[:, :self.n_bars]

    def set_fields(self, open, high, low, close, validity=None):
        """[n_symbols, n_bars] arrays; `validity`: optional dict field-index -> bool array (False = null)."""
        for f, a in enumerate((open, high, low, close)):
            a = np.ascontiguousarray(a, dtype=np.float64)
            assert a.shape == (self.n_symbols, self.n_bars)
            ok = None if validity is None else validity.get(f)
            if ok is None:
                self.host_field(f)[:] = a
            else:
                for s in range(self.n_symbols):
                    bits = np.packbits(np.asarray(ok[s], dtype=bool), bitorder="little")
                    N.check(N.lib().pqb_candles_set_column(self._h, s, f, a[s].ctypes.data_as(C.c_void_p),
                                                           bits.ctypes.data_as(C.c_void_p), 0, self.n_bars))

    def run_host(self, params: N.CandleParams | None = None):
        p = params or default_params(self.patterns_mask, self.prices_mask)
        N.check(N.lib().pqb_candles_run_host(self._h, C.byref(p)))

    def run(self, params: N.CandleParams | None = None):
        p = params or default_params(self.patterns_mask, self.prices_mask)
        N.check(N.lib().pqb_candles_run(self._h, C.byref(p)))

    def pattern(self, k: int) -> np.ndarray:
        """Int32 [n_symbols, n_bars] view of the host plane of pattern k (after run_host)."""
        return self._view(N.lib().pqb_candles_host_pattern(self._h, k), np.int32, self.pitch)[:, :self.n_bars]

    def price(self, k: int):
        """(values [n_symbols, n_bars], bool validity) of price output k (after run_host)."""
        v = self._view(N.lib().pqb_candles_host_price(self._h, k), np.float64, self.pitch)[:, :self.n_bars]
        w = self._view(N.lib().pqb_candles_host_price_validity(self._h, k), np.uint8, self.words_per_row * 4)
        ok = np.unpackbits(w, axis=1, bitorder="little")[:, :self.n_bars].astype(bool)
        return v, ok

    def fill_synthetic(self, seed: int = 1, to_host: bool = False):
        N.check(N.lib().pqb_candles_fill_synthetic(self._h, seed, 1 if to_host else 0))

    def fill_random_walk(self, seed: int = 0xC0FFEE, sigma: float = 0.02, to_host: bool = False):
        N.check(N.lib().pqb_candles_fill_random_walk(self._h, seed, sigma, 1 if to_host else 0))

    def time_device(self, params=None, warmup: int = 3, iters: int = 10) -> float:
        """Milliseconds of `iters` back-to-back fused candle launches on the device-resident panel."""
        p = params or default_params(self.patterns_mask, self.prices_mask)
        ms = C.c_float()
        N.check(N.lib().pqb_candles_time(self._h, C.byref(p), warmup, iters, C.byref(ms)))
        return float(ms.value)

    def live(self, params: N.CandleParams | None = None, max_push_bars: int = 64) -> "CandleLive":
        """A live candle panel primed from this panel's device inputs (run_host / fill_synthetic / fill_random_walk first).
        `params` (default: this panel's masks) chooses the outputs of the pushes, independently of this panel's planes."""
        return CandleLive(self, params, max_push_bars)


class CandleLive:
    """Append bars to a candle panel (include/pqb200.h "live candle panels").  Each push of k bars returns those k rows of
    every enabled pattern and price output, bit-identical to the last k rows of CandlePanel.run_host over the concatenated
    history.  Patterns and BOP refuse nulls (PqbError, PQB_ERR_NULLS); the price transforms propagate them.  commit=False
    previews a bar: the rows come back, the state stays.  The live panel keeps no reference to the candle panel."""
    FIELDS = ("open", "high", "low", "close")

    def __init__(self, cp: CandlePanel, params: N.CandleParams | None = None, max_push_bars: int = 64):
        self.params = params or default_params(cp.patterns_mask, cp.prices_mask)
        self.n_symbols = cp.n_symbols
        self.max_push_bars = int(max_push_bars)
        self.patterns = [k for k in range(N.N_PATTERNS) if self.params.patterns >> k & 1]
        self.prices = [k for k in range(N.N_PRICES) if self.params.prices >> k & 1]
        self.engine = cp.engine                     # (the native engine must outlive the live panel)
        self._h = C.c_void_p()
        N.check(N.lib().pqb_candles_live_create(cp._h, C.byref(self.params), C.c_int64(max_push_bars), C.byref(self._h)))
        names = pattern_names()
        self._pattern_names = {k: names[k] for k in self.patterns}

    def close(self):
        if self._h:
            N.lib().pqb_candles_live_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def bars(self) -> int:
        """History bars + committed bars."""
        return int(N.lib().pqb_candles_live_bars(self._h))

    def last_push_ms(self) -> float:
        """Device milliseconds of the last push (CUDA events from the copy of the new rows to the device to the end of the
        walk)."""
        ms = C.c_float()
        N.check(N.lib().pqb_candles_live_last_push_ms(self._h, C.byref(ms)))
        return ms.value

    def _rows(self, name, a, k, dtype=np.float64):
        a = np.asarray(a, dtype=dtype)
        if a.ndim == 1:
            a = a[None, :]
        if a.ndim != 2 or a.shape[1] != self.n_symbols:
            raise ValueError("%s has shape %r: expected [k, %d] or [%d]" % (name, a.shape, self.n_symbols, self.n_symbols))
        if k is not None and a.shape[0] != k:
            raise ValueError("%s has %d bars, expected %d" % (name, a.shape[0], k))
        return np.ascontiguousarray(a)

    def push(self, open=None, high=None, low=None, close=None, valid=None, commit: bool = True):
        """k new bars: each field float64 [k, n_symbols] (or [n_symbols] for one bar); a field no enabled output reads may
        be None.  `valid` None (all valid), one bool array for every field, or a dict {field: bool array} of the same shape.
        Returns ({pattern name: Int32 [n_symbols, k]}, {price name: (values, validity) [n_symbols, k]}) -- the orientation
        of CandlePanel.pattern() / .price()."""
        vals, k = {}, None
        for f, a in zip(self.FIELDS, (open, high, low, close)):
            if a is not None:
                vals[f] = self._rows(f, a, k)
                k = vals[f].shape[0]
        if k is None:
            raise ValueError("no field given")
        if k > self.max_push_bars:
            raise ValueError("%d bars in one push; this live candle panel takes at most %d" % (k, self.max_push_bars))
        masks = {}
        if valid is not None:
            per = valid if isinstance(valid, dict) else {f: valid for f in self.FIELDS}
            for f, m in per.items():
                if f not in self.FIELDS:
                    raise ValueError("unknown field %r in valid (open, high, low, close)" % (f,))
                masks[f] = np.packbits(self._rows("valid", m, k, bool), axis=1, bitorder="little")
        ptr = lambda a: None if a is None else a.ctypes.data_as(C.c_void_p)
        N.check(N.lib().pqb_candles_live_push(self._h, C.c_int64(k), *(ptr(vals.get(f)) for f in self.FIELDS),
                                              *(ptr(masks.get(f)) for f in self.FIELDS), 1 if commit else 0))
        n, vb = self.n_symbols, (self.n_symbols + 7) // 8
        pats, prices = {}, {}
        for p in self.patterns:
            a = np.ctypeslib.as_array((C.c_int32 * (k * n)).from_address(N.lib().pqb_candles_live_host_pattern(self._h, p)))
            pats[self._pattern_names[p]] = a.reshape(k, n).T.copy()
        for q in self.prices:
            v = np.ctypeslib.as_array((C.c_double * (k * n)).from_address(N.lib().pqb_candles_live_host_price(self._h, q)))
            b = np.ctypeslib.as_array((C.c_uint8 * (k * vb)).from_address(N.lib().pqb_candles_live_host_price_validity(self._h, q)))
            ok = np.unpackbits(b.reshape(k, vb), axis=1, bitorder="little")[:, :n].astype(bool)
            prices[N.PRICE_NAMES[q]] = (v.reshape(k, n).T.copy(), ok.T.copy())
        return pats, prices


def _col(a):
    a = np.ascontiguousarray(a, dtype=np.float64)
    return a, N.Col(a.ctypes.data_as(C.c_void_p), None, 0, a.size)


def cdl(pattern, open, high, low, close, penetration: float = 0.3, engine: Engine | None = None) -> np.ndarray:
    """One reference plugin call: pattern name or id on one symbol's columns -> Int32 array."""
    e = engine or get_engine(0)
    k = pattern if isinstance(pattern, int) else N.lib().pqb_pattern_index(pattern.encode())
    keep = [_col(x) for x in (open, high, low, close)]
    out = np.zeros(keep[0][0].size, dtype=np.int32)
    N.check(N.lib().pqb_cdl(e._h, k, *[C.byref(c) for _, c in keep], float(penetration), out.ctypes.data_as(C.c_void_p)))
    return out
