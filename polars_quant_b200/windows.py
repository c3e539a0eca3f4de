"""Many rolling windows in one launch (BASELINE config 5): KDJ(k) for several fastk windows, WILLR / MIDPRICE / Donchian(p)
for several windows and one ATR over a close / high / low panel (include/pqb200.h "many rolling windows", csrc/windows.cuh).

    wp = WindowPanel(10_000, 5_040, kdj=(5, 9, 14, 60, 250), ext=(5, 20, 55, 250), atr=14)
    wp.panel.set_fields(close=c, high=h, low=l)       # an ordinary Panel: set_column(s) / set_record_batch work too
    res = wp.compute()       # {"kdj_k_9": (values, validity), "kdj_d_9", "kdj_j_9", "willr_20", "midprice_20",
                             #  "donchian_upper_20", "donchian_lower_20", "atr_14", ...}

Replaces, per symbol, the reference's STOCH(h, l, c, k, 3, 0, 3, 0) (momentum.py:178-186; KDJ per SURVEY D3), willr
(momentum.rs:630), midprice (overlap.rs:281), atr (volatility.rs:18) called once per window; every value is bit-identical
to those calls.

Panels with halts, delistings, never-listed symbols or fields listed on different rows (validity bitmaps through
`panel.set_column(..., validity=)` / `set_columns`) follow the suite's null rules: each line equals, in values and validity,
what `Panel.compute` gives for the same single period.  A field is flagged at its first null after its own first valid bar.
- KDJ: fastk is valid where close is and the last k rows are valid in high and in low; slowk / slowd skip nulls; J is valid
  where D is.  Flags do not void KDJ.
- WILLR: all-null for a symbol flagged in close, high or low; otherwise valid where close, high and low are, after p - 1
  earlier bars with high and low valid.
- MIDPRICE / Donchian: all-null for a symbol flagged in high or low; otherwise valid where high and low are, the expanding
  window counting only such bars.
- ATR: the true range needs high, low and the previous row's close; the average counts valid true ranges.  Flags do not
  void ATR.
Symbol blocks without a flagged symbol run the plain kernel; the others run its null-aware variant beside it.

Live window panels: `wp.live(max_push_bars=64)` primes a `WindowLive` from the panel's device inputs; each
`push(close, high, low, valid=None, commit=True)` takes k new bars of every symbol and returns {name: (values [S, k],
validity [S, k])}, bit-identical to the last k rows of `compute()` over the concatenated history with the same validity.
Pushes may carry any validity pattern, under the null rules above applied per push: a first null after a field's first
valid bar flags it, and a new flag can turn a symbol's whole WILLR (close / high / low) or MIDPRICE / Donchian (high / low)
column null, history included -- `voided` names those columns after each push ({name: symbol indices}).  commit=False
previews a bar: the rows come back, the state stays.  The live panel keeps no reference to the window panel."""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _native as N
from .panel import Engine, Panel, get_engine

KDJ_LINES = ("kdj_k", "kdj_d", "kdj_j")
EXT_LINES = ("willr", "midprice", "donchian_upper", "donchian_lower")


class WindowPanel:
    def __init__(self, n_symbols: int, n_bars: int, kdj=(5, 9, 14, 60, 250), ext=(5, 20, 55, 250), atr: int = 14,
                 slowk_period: int = 3, slowd_period: int = 3, engine: Engine | None = None, host_staging: bool = True):
        self.engine = engine or get_engine(0)
        self.n_symbols, self.n_bars = int(n_symbols), int(n_bars)
        self.kdj, self.ext, self.atr = tuple(int(k) for k in kdj), tuple(int(p) for p in ext), int(atr or 0)
        ka = (C.c_int32 * max(1, len(self.kdj)))(*self.kdj)
        ea = (C.c_int32 * max(1, len(self.ext)))(*self.ext)
        self._h = C.c_void_p()
        N.check(N.lib().pqb_windows_create(self.engine._h, n_symbols, n_bars, ka, len(self.kdj), slowk_period, slowd_period, ea,
                                           len(self.ext), self.atr, 1 if host_staging else 0, C.byref(self._h)))
        n_slots = 3 * len(self.kdj) + 4 * len(self.ext) + (1 if self.atr else 0)
        self.panel = Panel._borrowed(N.lib().pqb_windows_panel(self._h), self.engine, n_symbols, n_bars, (1 << n_slots) - 1,
                                     host_staging, self)

    def close(self):
        if self._h:
            N.lib().pqb_windows_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def names(self):
        """{panel output slot: column name}"""
        out = {}
        for i, k in enumerate(self.kdj):
            for q, line in enumerate(KDJ_LINES):
                out[N.lib().pqb_windows_slot(self._h, 1, i, q)] = "%s_%d" % (line, k)
        for j, p in enumerate(self.ext):
            for q, line in enumerate(EXT_LINES):
                out[N.lib().pqb_windows_slot(self._h, 2, j, q)] = "%s_%d" % (line, p)
        if self.atr:
            out[N.lib().pqb_windows_slot(self._h, 3, 0, 0)] = "atr_%d" % self.atr
        return out

    def run(self):
        N.check(N.lib().pqb_windows_run(self._h))

    def compute(self):
        self.panel.upload()
        self.run()
        self.panel.download()
        self.panel.sync()
        return {name: (self.panel.host_output(k), self.panel.host_validity(k)) for k, name in self.names().items()}

    def fill_synthetic(self, seed: int = 55, sigma: float = 0.02, to_host: bool = False):
        self.panel.fill_synthetic(seed=seed, sigma=sigma, to_host=to_host)

    def time_device(self, warmup: int = 2, iters: int = 5):
        ms = C.c_float()
        N.check(N.lib().pqb_windows_time(self._h, warmup, iters, C.byref(ms)))
        return ms.value / iters, N.lib().pqb_windows_last_launches(self._h)

    def live(self, max_push_bars: int = 64) -> "WindowLive":
        """A live window panel primed from this panel's device inputs (compute / upload / fill_synthetic first)."""
        return WindowLive(self, max_push_bars)


class WindowLive:
    """Append bars to a many-window panel (include/pqb200.h "live window panels"); see the module docstring."""
    FIELDS = ("close", "high", "low")

    def __init__(self, wp: WindowPanel, max_push_bars: int = 64):
        self.n_symbols = wp.n_symbols
        self.max_push_bars = int(max_push_bars)
        self.names = wp.names()                     # {slot: name}
        self.voided = {}                            # (the last push's; a new dict per push)
        self.engine = wp.engine                     # (the native engine must outlive the live panel)
        self._h = C.c_void_p()
        N.check(N.lib().pqb_windows_live_create(wp._h, C.c_int64(max_push_bars), C.byref(self._h)))

    def close(self):
        if self._h:
            N.lib().pqb_windows_live_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def bars(self) -> int:
        """History bars + committed bars."""
        return int(N.lib().pqb_windows_live_bars(self._h))

    @property
    def state_bytes(self) -> int:
        return int(N.lib().pqb_windows_live_state_bytes(self._h))

    def last_push_ms(self) -> float:
        """Device milliseconds of the last push (CUDA events from the pack of the new rows to the unpack of the results)."""
        ms = C.c_float()
        N.check(N.lib().pqb_windows_live_last_push_ms(self._h, C.byref(ms)))
        return ms.value

    def _rows(self, name, a, k, dtype=np.float64):
        if a is None:
            raise ValueError("%s is required" % name)
        a = np.asarray(a, dtype=dtype)
        if a.ndim == 1:
            a = a[None, :]
        if a.ndim != 2 or a.shape[1] != self.n_symbols:
            raise ValueError("%s has shape %r: expected [k, %d] or [%d]" % (name, a.shape, self.n_symbols, self.n_symbols))
        if k is not None and a.shape[0] != k:
            raise ValueError("%s has %d bars, close has %d" % (name, a.shape[0], k))
        return np.ascontiguousarray(a)

    def push(self, close, high, low, valid=None, commit: bool = True):
        """k new bars: close / high / low float64 [k, n_symbols] (or [n_symbols] for one bar); `valid` None (all valid), one
        bool array for every field, or a dict {field: bool array} of the same shape.  Returns {name: (values, validity)} of
        shape [n_symbols, k] and sets `voided`: {name: indices of the symbols whose earlier rows of that line this push
        turned null} (a preview's too)."""
        c = self._rows("close", close, None)
        k = c.shape[0]
        if k > self.max_push_bars:
            raise ValueError("%d bars in one push; this live window panel takes at most %d" % (k, self.max_push_bars))
        vals = {"close": c, "high": self._rows("high", high, k), "low": self._rows("low", low, k)}
        masks = {}
        if valid is not None:
            per = valid if isinstance(valid, dict) else {f: valid for f in self.FIELDS}
            for f, m in per.items():
                if f not in self.FIELDS:
                    raise ValueError("unknown field %r in valid (close, high, low)" % (f,))
                masks[f] = np.packbits(self._rows("valid", m, k, bool), axis=1, bitorder="little")
        ptr = lambda a: None if a is None else a.ctypes.data_as(C.c_void_p)
        N.check(N.lib().pqb_windows_live_push(self._h, C.c_int64(k), *(ptr(vals[f]) for f in self.FIELDS),
                                              *(ptr(masks.get(f)) for f in self.FIELDS), 1 if commit else 0))
        vb = (self.n_symbols + 7) // 8
        res, voided = {}, {}
        for slot, name in self.names.items():
            vp = N.lib().pqb_windows_live_host_output(self._h, slot)
            bp = N.lib().pqb_windows_live_host_validity(self._h, slot)
            v = np.ctypeslib.as_array((C.c_double * (k * self.n_symbols)).from_address(vp)).reshape(k, self.n_symbols)
            b = np.ctypeslib.as_array((C.c_uint8 * (k * vb)).from_address(bp)).reshape(k, vb)
            ok = np.unpackbits(b, axis=1, bitorder="little")[:, :self.n_symbols].astype(bool)
            res[name] = (v.T.copy(), ok.T.copy())
            w = np.ctypeslib.as_array((C.c_uint8 * vb).from_address(N.lib().pqb_windows_live_host_voided(self._h, slot)))
            syms = np.flatnonzero(np.unpackbits(w, bitorder="little")[:self.n_symbols])
            if len(syms):
                voided[name] = syms
        self.voided = voided
        return res
