"""Runs the reference's plugin functions from their own source text.  TEST INFRASTRUCTURE.

`Reference()` parses src/talib/{overlap,momentum,volatility,volume,price,pattern}.rs of the original and
exposes `call(fn_name, columns, params=..., kwargs=...)`, which builds the `inputs: &[Series]` (+ the serde
kwargs struct) exactly as polars would hand them to `#[polars_expr] fn <fn_name>` and returns the result
columns as (values, validity) numpy pairs -- or raises `ReferenceError` (a `PolarsResult::Err`) /
`ReferencePanic` (a Rust panic: process abort under the crate's `panic = "abort"`).

What is NOT the reference's text (frozen decisions of SURVEY.md 8a, restated here and nowhere else):
* D1 `calc_rma`: called by momentum.rs:21,42,379,434,526,527,701-703 but defined nowhere in the snapshot.
  Defined as the Wilder smoothing in calc_ema's own structure: None for i < p-1, out[p-1] = (sum of the
  first p values, left to right) / p, then out[i] = (1/p).mul_add(x[i] - out[i-1], out[i-1]).
* D2: momentum.rs passes slices to overlap's calc_ema / calc_sma and indexes the result like a
  Vec<Option<f64>>; the adapter in rs_eval.Interp.call_fn presents the slice as a null-free Float64Chunked
  to the callee's own text and gives the result list access.  No arithmetic involved.
"""
from __future__ import annotations

from pathlib import Path

import numpy as np

from . import polars_model as M
from . import reference_root
from .polars_model import Err, Ok, RustPanic, Some
from .rs_eval import Interp, RustRuntimeError
from .rs_parse import parse_rust

MODULES = ("overlap", "momentum", "volatility", "volume", "price", "pattern")


class ReferenceError(Exception):
    """The reference returns PolarsResult::Err (e.g. cont_slice() on a column with nulls)."""


class ReferencePanic(Exception):
    """The reference panics (abort)."""


def calc_rma(x, p):
    """D1 (see module docstring)."""
    n = len(x)
    out = [None] * n
    if p == 0 or n < p:
        return out
    s = 0.0
    for j in range(p):
        s += x[j]
    prev = M.fdiv(s, float(p))
    out[p - 1] = Some(prev)
    alpha = 1.0 / float(p)
    for i in range(p, n):
        prev = M.fma(alpha, x[i] - prev, prev)
        out[i] = Some(prev)
    return out


def series(values, validity=None, chunks=None, dtype="Float64", force_bitmap=False):
    """numpy column -> model Series.  `chunks`: list of chunk lengths (default: one chunk).
    `force_bitmap`: give every chunk a validity bitmap even when it has no nulls (legal Arrow; selects the
    reference's `Some(bitmap)` branches on dense data)."""
    vals = [float(v) for v in values] if dtype == "Float64" else [int(v) for v in values]
    n = len(vals)
    valid = None if validity is None else [bool(b) for b in validity]
    bounds = [0]
    for c in (chunks or [n]):
        bounds.append(bounds[-1] + c)
    assert bounds[-1] == n, "chunk lengths must add up"
    out = []
    for a, b in zip(bounds[:-1], bounds[1:]):
        v = None if valid is None else valid[a:b]
        if v is not None and all(v) and not force_bitmap:
            v = None
        if v is None and force_bitmap:
            v = [True] * (b - a)
        out.append(M.PrimArray(vals[a:b], v))
    return M.Series(M.ChunkedArray("", out, dtype))


def literal(v):
    """A trailing parameter as the Rust signature reads it: `.i64()` for ints, `.f64()` for floats."""
    if isinstance(v, float):
        return M.Series(M.ChunkedArray.from_values("literal", [v], "Float64"))
    return M.Series(M.ChunkedArray.from_values("literal", [int(v)], "Int64"))


def column(ca):
    items = ca.opt_items()
    ok = np.array([it is not None for it in items], dtype=bool)
    if ca.dtype == "Float64":
        vals = np.array([np.nan if it is None else it.v for it in items], dtype=np.float64)
    else:
        vals = np.array([0 if it is None else it.v for it in items], dtype=np.int64)
    return vals, ok


class Reference:
    def __init__(self, src: Path | None = None, modules=MODULES):
        src = src or reference_root() / "src" / "talib"
        self.interp = Interp()
        self.interp.extern["calc_rma"] = calc_rma
        self.where = {}
        for m in modules:
            parsed = parse_rust((src / f"{m}.rs").read_text(), f"{m}.rs")
            self.interp.load(m, parsed)
            for name, node in parsed["fns"].items():
                self.where.setdefault(name, (m, node[5]))
        self.kwargs_struct = {}
        for m in modules:
            for name, fn in self.interp.modules[m].fns.items():
                params = fn.node[2]
                if len(params) == 2 and params[1][1][0] == "path":
                    self.kwargs_struct[name] = (m, params[1][1][1])

    def functions(self):
        return sorted(self.where)

    def raw(self, fn, *args):
        m, _ = self.where[fn]
        try:
            return self.interp.call(m, fn, *args)
        except RustPanic as e:
            raise ReferencePanic(str(e)) from None

    def call(self, fn, columns, params=(), kwargs=None):
        """columns: list of Series (see `series`); params: trailing literal inputs; kwargs: dict for the serde
        struct of functions declared `fn f(inputs, kwargs: K)`.  Returns a list of (values, validity)."""
        inputs = list(columns) + [literal(p) for p in params]
        args = [inputs]
        if fn in self.kwargs_struct:
            m, sname = self.kwargs_struct[fn]
            args.append(self.interp.make_struct(m, sname, **(kwargs or {})))
        elif kwargs:
            raise TypeError(f"{fn} takes no kwargs")
        res = self.raw(fn, *args)
        if isinstance(res, Err):
            raise ReferenceError(res.v)
        if not isinstance(res, Ok):
            raise RustRuntimeError(f"{fn} returned {type(res).__name__}")
        s = res.v
        inner = s.inner
        if isinstance(inner, M.StructChunked):
            return [column(f.inner) for f in inner.fields]
        return [column(inner)]
