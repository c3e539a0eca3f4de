"""Live panels (include/pqb200.h "live panels"): a panel's history is computed once, then every new bar of every symbol
is appended with a push that returns only the new rows -- bit-identical, values and validity, to the last rows of a full
recompute over the concatenated history.

    panel = Panel(n_symbols, n_bars); panel.set_fields(...); full = panel.compute()
    live = LivePanel(panel)
    rows = live.push(close, high, low, volume)     # {name: (values [n_symbols, k], validity [n_symbols, k])}

`full[name][0][:, T:T + k]` of a recompute over T + k bars equals `rows[name][0]`.  push(..., commit=False) previews the
current, unfinished bar: the rows come back, the state and `bars` stay as they were.

LivePanel(panel, nulls=True) accepts histories with halts, delistings and fields listed on different rows, and pushes
with any validity pattern.  A null after a field's first valid bar turns the symbol's whole column of macd / rsi / willr /
midprice (...) null in the reference, history included; after each push `voided` names the columns it did that to:
{output name: symbol indices}.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _native as N


class LivePanel:
    FIELDS = ("close", "high", "low", "volume")
    nulls = False
    voided: dict = {}                               # (the last push's; a new dict per push)

    def __init__(self, panel, params: N.SuiteParams | None = None, outputs: int | None = None, max_push_bars: int = 64,
                 nulls: bool = False):
        """`panel`: a Panel whose inputs are on the device (compute / upload / run_host / fill_synthetic).  `outputs`: a
        mask of output ids (None: the outputs of params.indicators).  `nulls`: the null-aware live panel (any validity
        pattern in the history and the pushes; see `voided`).  The live panel keeps no reference to `panel`."""
        if not isinstance(nulls, (bool, np.bool_)):
            raise TypeError("nulls must be True or False, not %r" % (nulls,))
        self.params = params or N.default_params()
        self.n_symbols = panel.n_symbols
        self.max_push_bars = int(max_push_bars)
        self.nulls = bool(nulls)
        self.voided = {}
        self.engine = panel.engine                  # (the native engine must outlive the live panel)
        self._h = C.c_void_p()
        N.check(N.lib().pqb_live_create_ex(panel._h, C.byref(self.params), C.c_uint64(outputs or 0), C.c_int64(max_push_bars),
                                           C.c_uint32(N.LIVE_NULLS if self.nulls else 0), C.byref(self._h)))
        self.outputs = [k for k in range(N.N_OUTPUTS) if N.lib().pqb_live_host_output(self._h, k)]

    def close(self):
        if self._h:
            N.lib().pqb_live_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def bars(self) -> int:
        """History bars + committed bars."""
        return int(N.lib().pqb_live_bars(self._h))

    @property
    def state_bytes(self) -> int:
        return int(N.lib().pqb_live_state_bytes(self._h))

    def last_push_ms(self) -> float:
        """Device milliseconds of the last push (CUDA events from the pack of the new rows to the unpack of the results)."""
        ms = C.c_float()
        N.check(N.lib().pqb_live_last_push_ms(self._h, C.byref(ms)))
        return ms.value

    def _rows(self, name, a, k):
        a = np.asarray(a, dtype=np.float64 if name != "valid" else bool)
        if a.ndim == 1:
            a = a[None, :]
        if a.ndim != 2 or a.shape[1] != self.n_symbols:
            raise ValueError("%s has shape %r: expected [k, %d] or [%d]" % (name, a.shape, self.n_symbols, self.n_symbols))
        if k is not None and a.shape[0] != k:
            raise ValueError("%s has %d bars, close has %d" % (name, a.shape[0], k))
        return np.ascontiguousarray(a)

    def push(self, close, high=None, low=None, volume=None, valid=None, commit: bool = True):
        """k new bars: each field float64 [k, n_symbols] (or [n_symbols] for one bar); `valid` None (all valid), one bool
        array for every field, or a dict {field: bool array} of the same shape.  Returns {name: (values, validity)} of
        shape [n_symbols, k] -- the orientation of Panel.outputs().  Null-aware panels also set `voided`: {output name:
        indices of the symbols whose earlier rows of that output this push turned null} (a preview's too)."""
        c = self._rows("close", close, None)
        k = c.shape[0]
        if k > self.max_push_bars:
            raise ValueError("%d bars in one push; this live panel takes at most %d" % (k, self.max_push_bars))
        vals = {"close": c}
        for name, a in (("high", high), ("low", low), ("volume", volume)):
            if a is not None:
                vals[name] = self._rows(name, a, k)
        masks = {}
        if valid is not None:
            per = valid if isinstance(valid, dict) else {f: valid for f in self.FIELDS}
            for f, m in per.items():
                if f not in self.FIELDS:
                    raise ValueError("unknown field %r in valid" % (f,))
                m = self._rows("valid", m, k)
                masks[f] = np.packbits(m, axis=1, bitorder="little")
        ptr = lambda a: None if a is None else a.ctypes.data_as(C.c_void_p)
        N.check(N.lib().pqb_live_push(self._h, C.c_int64(k), *(ptr(vals.get(f)) for f in self.FIELDS),
                                      *(ptr(masks.get(f)) for f in self.FIELDS), 1 if commit else 0))
        vb = (self.n_symbols + 7) // 8
        res = {}
        for kk in self.outputs:
            vp = N.lib().pqb_live_host_output(self._h, kk)
            bp = N.lib().pqb_live_host_validity(self._h, kk)
            v = np.ctypeslib.as_array((C.c_double * (k * self.n_symbols)).from_address(vp)).reshape(k, self.n_symbols)
            b = np.ctypeslib.as_array((C.c_uint8 * (k * vb)).from_address(bp)).reshape(k, vb)
            ok = np.unpackbits(b, axis=1, bitorder="little")[:, :self.n_symbols].astype(bool)
            res[N.OUTPUT_NAMES[kk]] = (v.T.copy(), ok.T.copy())
        voided = {}
        if self.nulls:
            for kk in self.outputs:
                b = np.ctypeslib.as_array((C.c_uint8 * vb).from_address(N.lib().pqb_live_host_voided(self._h, kk)))
                syms = np.flatnonzero(np.unpackbits(b, bitorder="little")[:self.n_symbols])
                if len(syms):
                    voided[N.OUTPUT_NAMES[kk]] = syms
        self.voided = voided
        return res
