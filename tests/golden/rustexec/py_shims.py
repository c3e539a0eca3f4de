"""Imports the reference's Python shim modules (python/polars_quant/talib/*.py) VERBATIM and runs them on top
of the executed Rust text.  TEST INFRASTRUCTURE.

polars is not installable here, so `import polars as pl` / `from polars.plugins import
register_plugin_function` inside the shims resolve to the minimal eager stand-ins below:

* `register_plugin_function(args=[exprs..., literals...], function_name=f)` calls the reference's Rust
  `fn f` (rustexec.ref_exec.Reference).  Two intent mappings, because the literal Python -> Rust hand-over is
  broken in the snapshot (SURVEY.md section 5, "Config / flags"): (1) for Rust functions declared
  `fn f(inputs, kwargs: K)` the positional literals become K's fields in declaration order (the shims never
  pass `kwargs=`, which pyo3-polars would reject); (2) integer literals arrive as Int64 (polars makes Int32
  literals, on which the Rust `.i64()?` is an Err).
* `Expr.rolling_min(k)` / `rolling_max(k)`: polars 1.39 semantics with the defaults the shims use
  (`min_samples = window_size`, no weights, not centred): null until k values are in the window and
  wherever the window holds a null; otherwise the min / max of the k values (NaN-free data only: polars'
  NaN ordering inside rolling windows is not modelled).
* `+ - * /` between expressions / scalars: polars' null-propagating element-wise IEEE arithmetic.
* `.alias()`, `.struct.field()`: naming only.
"""
from __future__ import annotations

import importlib
import sys
import types

from . import polars_model as M
from . import reference_root
from .polars_model import Some
from .ref_exec import Reference, column, literal


class Expr:
    """An eagerly evaluated expression: one column (ChunkedArray) or a struct of named columns."""

    def __init__(self, ca=None, fields=None):
        self.ca, self.fields = ca, fields

    # arithmetic
    def _bin(self, op, other, swap=False):
        b = other.ca if isinstance(other, Expr) else other
        a = self.ca
        return Expr(M.chunked_binop(op, b, a) if swap else M.chunked_binop(op, a, b))

    def __add__(self, o): return self._bin("+", o)
    def __sub__(self, o): return self._bin("-", o)
    def __mul__(self, o): return self._bin("*", o)
    def __truediv__(self, o): return self._bin("/", o)
    def __radd__(self, o): return self._bin("+", o, True)
    def __rsub__(self, o): return self._bin("-", o, True)
    def __rmul__(self, o): return self._bin("*", o, True)
    def __rtruediv__(self, o): return self._bin("/", o, True)

    def alias(self, _name):
        return self

    def _rolling(self, k, pick):
        items = self.ca.opt_items()
        out = []
        for i in range(len(items)):
            if i + 1 < k:
                out.append(None)
                continue
            w = items[i + 1 - k:i + 1]
            if any(x is None for x in w):
                out.append(None)
                continue
            vals = [x.v for x in w]
            assert all(v == v for v in vals), "rolling_min/max over NaN values is not modelled"
            out.append(Some(pick(vals)))
        return Expr(M.ChunkedArray.from_options("", out))

    def rolling_min(self, window_size):
        return self._rolling(window_size, min)

    def rolling_max(self, window_size):
        return self._rolling(window_size, max)

    @property
    def struct(self):
        return _StructNs(self)

    def numpy(self):
        return column(self.ca)


class _StructNs:
    def __init__(self, e):
        self.e = e

    def field(self, name):
        return Expr(self.e.fields[name])


class Shims:
    """`Shims().talib.momentum.STOCH(high, low, close, ...)` with `Expr` inputs."""

    def __init__(self, ref: Reference | None = None):
        self.ref = ref or Reference()
        pl = types.ModuleType("polars")
        pl.Expr = Expr
        pl.Series = type("Series", (), {})          # never an input type here: the shims return the expression
        pl.DataFrame = type("DataFrame", (), {})
        plugins = types.ModuleType("polars.plugins")
        plugins.register_plugin_function = self._register
        pl.plugins = plugins
        saved = {k: sys.modules.get(k) for k in ("polars", "polars.plugins")}
        sys.modules["polars"], sys.modules["polars.plugins"] = pl, plugins
        try:
            ref_py = reference_root() / "python" / "polars_quant"
            pkg = types.ModuleType("_refpq")
            pkg.__path__ = [str(ref_py)]
            talib = types.ModuleType("_refpq.talib")
            talib.__path__ = [str(ref_py / "talib")]
            sys.modules["_refpq"], sys.modules["_refpq.talib"] = pkg, talib
            for m in ("overlap", "momentum", "volatility", "volume", "price"):
                setattr(talib, m, importlib.import_module(f"_refpq.talib.{m}"))
            self.talib = talib
        finally:
            for k, v in saved.items():
                if v is None:
                    sys.modules.pop(k, None)
                else:
                    sys.modules[k] = v

    def _register(self, args, plugin_path=None, function_name=None, is_elementwise=False, **_):
        ref = self.ref
        cols = [a for a in args if isinstance(a, Expr)]
        lits = [a for a in args if not isinstance(a, Expr)]
        inputs = [M.Series(c.ca) for c in cols]
        call_args = [inputs]
        if function_name in ref.kwargs_struct:
            m, sname = ref.kwargs_struct[function_name]
            names = ref.interp.modules[m].structs[sname]
            call_args.append(ref.interp.make_struct(m, sname, **dict(zip(names, lits))))
        else:
            inputs.extend(literal(v) for v in lits)
        res = ref.raw(function_name, *call_args)
        if isinstance(res, M.Err):
            from .ref_exec import ReferenceError
            raise ReferenceError(res.v)
        inner = res.v.inner
        if isinstance(inner, M.StructChunked):
            return Expr(fields={f.inner.name: f.inner for f in inner.fields})
        return Expr(inner)


def expr(values, validity=None):
    from .ref_exec import series
    return Expr(series(values, validity).inner)
