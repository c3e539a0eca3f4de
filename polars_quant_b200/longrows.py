"""Few symbols, very long rows (BASELINE config 3: 500 symbols x 1,000,000 minute bars): several EMA periods and the
MACD in ONE pass over close, parallel along time (include/pqb200.h "long rows", csrc/longrows.cuh).

    lp = LongPanel(500, 1_000_000, ema_periods=(12, 26, 200, 5000), macd=(12, 26, 9))
    lp.panel.set_fields(close=close)            # or set_column / set_columns / set_record_batch: an ordinary Panel
    res = lp.compute()                          # {"ema_12": (values, validity), ..., "macd": ..., "macd_signal": ..., "macd_hist": ...}

Replaces, per symbol, `with_columns([EMA(c, 12), EMA(c, 26), EMA(c, 200), EMA(c, 5000), *MACD(c, 12, 26, 9)])` of the
reference (README.md:1360-1365): calc_ema overlap.rs:660-730, macd momentum.rs:250-283.  Tolerance-exact, like SplitPanel
but with no warm-up: the EMA lines within rel 1e-10 / abs 1e-12 of the serial reference, the MACD lines (which cross zero)
within that plus 4 ulp of the row's largest |close|; the first time tile is bit-exact."""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _native as N
from .panel import Engine, Panel, get_engine

MACD_SLOTS = (7, 8, 9)          # enum pqb_output: macd, macd_signal, macd_hist


class LongPanel:
    def __init__(self, n_symbols: int, n_bars: int, ema_periods=(12, 26, 200, 5000), macd=(12, 26, 9),
                 engine: Engine | None = None, tile_bars: int = 0, host_staging: bool = True):
        self.engine = engine or get_engine(0)
        self.n_symbols, self.n_bars = int(n_symbols), int(n_bars)
        self.ema_periods = tuple(int(p) for p in ema_periods)
        self.macd = tuple(int(p) for p in macd) if macd else (0, 0, 0)
        self._periods = (C.c_int32 * max(1, len(self.ema_periods)))(*self.ema_periods)
        self._h = C.c_void_p()
        N.check(N.lib().pqb_long_create(self.engine._h, n_symbols, n_bars, len(self.ema_periods), 1 if macd else 0, tile_bars,
                                        1 if host_staging else 0, C.byref(self._h)))
        om = (1 << len(self.ema_periods)) - 1
        if macd:
            om |= 7 << 7
        self.panel = Panel._borrowed(N.lib().pqb_long_panel(self._h), self.engine, n_symbols, n_bars, om, host_staging, self)

    def close(self):
        if self._h:
            N.lib().pqb_long_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def names(self):
        out = {k: "ema_%d" % p for k, p in enumerate(self.ema_periods)}
        if any(self.macd):
            out.update(dict(zip(MACD_SLOTS, ("macd", "macd_signal", "macd_hist"))))
        return out

    def run(self):
        """Device-resident (close already uploaded); asynchronous."""
        N.check(N.lib().pqb_long_run(self._h, self._periods, len(self.ema_periods), *self.macd))

    def compute(self):
        """upload + run + download + sync -> {name: (values [n_symbols, n_bars], validity)}."""
        self.panel.upload()
        self.run()
        self.panel.download()
        self.panel.sync()
        return {name: (self.panel.host_output(k), self.panel.host_validity(k)) for k, name in self.names().items()}

    def fill_synthetic(self, seed: int = 3, sigma: float = 0.0005, to_host: bool = False):
        self.panel.fill_synthetic(seed=seed, sigma=sigma, to_host=to_host)

    def time_device(self, warmup: int = 2, iters: int = 5):
        """(milliseconds per pass, kernel launches per pass), CUDA events on the engine's stream."""
        ms = C.c_float()
        N.check(N.lib().pqb_long_time(self._h, self._periods, len(self.ema_periods), *self.macd, warmup, iters, C.byref(ms)))
        return ms.value / iters, N.lib().pqb_long_last_launches(self._h)
