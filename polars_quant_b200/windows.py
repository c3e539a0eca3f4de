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
Symbol blocks without a flagged symbol run the plain kernel; the others run its null-aware variant beside it."""
from __future__ import annotations

import ctypes as C

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
