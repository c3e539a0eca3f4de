"""Wide `{symbol}_{column}` panels: the data format on both sides of the hot path (SURVEY.md 8f.4).

The reference documents its panel format only in README.md:88-161: `load(folder, file_type, prefix, suffix,
has_header)` reads one file per symbol (file name = symbol, a `date` column required), full-joins them on `date`
and returns a DataFrame whose first column is `date` and whose other columns are `{symbol}_{column}`
(`AAPL_open`, `AAPL_close`, ...).  Its indicator engine is then applied column by column through polars.
Here the same wide table (pyarrow; polars is not in this image) goes to the GPU as ONE panel:

    table = load("data/stocks", file_type=["parquet"])
    wp = WidePanel(table)                       # {symbol}_{open,high,low,close,volume} -> device panel(s)
    out = wp.suite()                            # date + {symbol}_{sma,ema,...,midprice}: 21 columns per symbol
    cdl = wp.candles()                          # date + {symbol}_{cdl2crows,...,bop}

Arrow validity goes in as is (a symbol listed later has leading nulls, a halt has interior nulls: the engine's
null rules apply, DESIGN.md section 5); results come back as Arrow arrays that alias the panel's pinned host
buffers (zero copy; they keep the panel alive).
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

import numpy as np
import pyarrow as pa
import pyarrow.compute as pc

from . import _native as N
from .candles import CandlePanel, default_params as candle_default_params, pattern_names
from .panel import Engine, Panel, get_engine

SUITE_FIELDS = ("close", "high", "low", "volume")          # enum pqb_field order
CANDLE_FIELDS = ("open", "high", "low", "close")           # enum pqb_candle_field order
_READERS = ("parquet", "csv", "json", "feather", "ipc")    # (xlsx / xls of the README need a spreadsheet reader: not in this image)


def _read(path: Path, kind: str, has_header: bool) -> pa.Table:
    if kind == "parquet":
        import pyarrow.parquet as pq
        return pq.read_table(path)
    if kind == "csv":
        import pyarrow.csv as pcsv
        ro = pcsv.ReadOptions(autogenerate_column_names=not has_header)
        return pcsv.read_csv(path, read_options=ro)
    if kind == "json":
        import pyarrow.json as pjson
        return pjson.read_json(path)
    import pyarrow.feather as pf
    return pf.read_table(path)


def load(folder, file_type=None, prefix=None, suffix=None, has_header: bool = True) -> pa.Table:
    """README.md:90-161 `load`: every file of `folder` with one of the `file_type` extensions (default: all supported)
    whose stem starts with `prefix` / ends with `suffix` is one symbol (symbol = file stem); all are full-joined on
    `date` (sorted ascending) into `date`, `{symbol}_{column}`..."""
    folder = Path(folder)
    kinds = [k.lower() for k in (file_type or _READERS)]
    for k in kinds:
        if k in ("xlsx", "xls"):
            raise NotImplementedError("spreadsheet files need a reader that is not in this image")
        if k not in _READERS:
            raise ValueError("unsupported file type %r" % k)
    files = sorted(p for p in folder.iterdir() if p.is_file() and p.suffix[1:].lower() in kinds
                   and (prefix is None or p.stem.startswith(prefix)) and (suffix is None or p.stem.endswith(suffix)))
    if not files:
        raise FileNotFoundError("no matching files in %s" % folder)
    per_symbol = {}
    for p in files:
        t = _read(p, p.suffix[1:].lower(), has_header)
        if "date" not in t.column_names:
            raise ValueError("%s has no `date` column" % p.name)
        per_symbol[p.stem] = t
    dates = pa.chunked_array([t["date"].combine_chunks().cast(next(iter(per_symbol.values()))["date"].type)
                              for t in per_symbol.values()])
    all_dates = pc.unique(dates.combine_chunks())
    all_dates = all_dates.take(pc.sort_indices(all_dates))
    cols, names = [all_dates], ["date"]
    for sym, t in per_symbol.items():
        idx = pc.index_in(all_dates, value_set=t["date"].combine_chunks().cast(all_dates.type))   # null where the symbol has no row
        for name in t.column_names:
            if name == "date":
                continue
            cols.append(t[name].combine_chunks().take(idx))
            names.append("%s_%s" % (sym, name))
    return pa.table(cols, names=names)


def prepare_sequential_data(folder_path, date_col: str = "date", symbol_col: str = "symbol", fill_null_strategy: str = "forward",
                            default_fill_value: float = 0.0) -> pa.Table:
    """python/polars_quant/backtest/sequential.py:7-93 over pyarrow: every .csv / .parquet / .pqt file of the folder (the
    file stem is the symbol when the file has no `symbol_col`) is concatenated (union of the columns), aligned on the
    full `unique dates x unique symbols` grid, sorted by (date, symbol), and its value columns are filled per symbol
    ("forward", "backward" or "zero") and then with `default_fill_value` (what is still null, e.g. before a listing).
    Returns the LONG table `date_col, symbol_col, value columns...`; `to_wide` pivots it into a `{symbol}_{column}` panel.
    Value columns must be numeric (they come back as Float64); a (date, symbol) pair may appear only once."""
    folder = Path(folder_path)
    if not folder.exists() or not folder.is_dir():
        raise FileNotFoundError("The directory '%s' does not exist or is not a directory." % folder_path)
    frames = []
    for p in sorted(folder.iterdir()):
        ext = p.suffix.lower()
        if ext == ".csv":
            t = _read(p, "csv", True)
        elif ext in (".parquet", ".pqt"):
            t = _read(p, "parquet", True)
        else:
            continue
        if symbol_col not in t.column_names:
            t = t.append_column(symbol_col, pa.array([p.stem] * t.num_rows, type=pa.string()))
        frames.append(t)
    if not frames:
        raise ValueError("No valid CSV or Parquet files found in '%s'." % folder_path)
    value_cols = []
    for t in frames:
        value_cols += [c for c in t.column_names if c not in (date_col, symbol_col) and c not in value_cols]
    date_type = frames[0][date_col].type
    dates = pa.concat_arrays([t[date_col].combine_chunks().cast(date_type) for t in frames])
    syms = pa.concat_arrays([t[symbol_col].combine_chunks().cast(pa.string()) for t in frames])
    u_dates = pc.unique(dates)
    u_dates = u_dates.take(pc.sort_indices(u_dates))
    u_syms = pc.unique(syms)
    u_syms = u_syms.take(pc.sort_indices(u_syms))
    nd, ns = len(u_dates), len(u_syms)
    di = np.asarray(pc.index_in(dates, value_set=u_dates).to_numpy(zero_copy_only=False), dtype=np.int64)
    si = np.asarray(pc.index_in(syms, value_set=u_syms).to_numpy(zero_copy_only=False), dtype=np.int64)
    cell = di * ns + si
    if len(np.unique(cell)) != len(cell):
        raise ValueError("a (%s, %s) pair appears more than once" % (date_col, symbol_col))
    out_cols = [u_dates.take(pa.array(np.repeat(np.arange(nd), ns))), u_syms.take(pa.array(np.tile(np.arange(ns), nd)))]
    row0 = np.cumsum([0] + [t.num_rows for t in frames])
    for name in value_cols:
        grid = np.full(nd * ns, np.nan)
        have = np.zeros(nd * ns, dtype=bool)
        for k, t in enumerate(frames):
            if name not in t.column_names:
                continue
            a = _f64(t[name])
            ok = ~np.asarray(a.is_null())
            idx = cell[row0[k]:row0[k + 1]][ok]
            grid[idx] = np.asarray(a.to_numpy(zero_copy_only=False), dtype=np.float64)[ok]
            have[idx] = True
        grid, have = grid.reshape(nd, ns), have.reshape(nd, ns)
        if fill_null_strategy in ("forward", "backward"):
            rows = np.arange(nd)[:, None]
            if fill_null_strategy == "forward":
                src = np.maximum.accumulate(np.where(have, rows, -1), axis=0)               # last valid row at or before
                okf = src >= 0
            else:
                src = np.minimum.accumulate(np.where(have, rows, nd)[::-1], axis=0)[::-1]   # first valid row at or after
                okf = src < nd
            grid = np.where(okf, np.take_along_axis(grid, np.clip(src, 0, nd - 1), axis=0), np.nan)
            have = okf
        elif fill_null_strategy == "zero":
            grid, have = np.where(have, grid, 0.0), np.ones_like(have)
        grid = np.where(have, grid, float(default_fill_value))
        out_cols.append(pa.array(grid.reshape(-1)))
    return pa.table(out_cols, names=[date_col, symbol_col] + value_cols)


def to_wide(long_table: pa.Table, date_col: str = "date", symbol_col: str = "symbol") -> pa.Table:
    """Long (date, symbol, values...) -> the wide `date`, `{symbol}_{column}` panel of README.md:88-161 (what `load`
    returns and `WidePanel` takes); (date, symbol) pairs that are absent become nulls."""
    dates = long_table[date_col].combine_chunks()
    syms = long_table[symbol_col].combine_chunks().cast(pa.string())
    u_dates = pc.unique(dates)
    u_dates = u_dates.take(pc.sort_indices(u_dates))
    u_syms = pc.unique(syms)                                                              # order of first appearance
    di = np.asarray(pc.index_in(dates, value_set=u_dates).to_numpy(zero_copy_only=False), dtype=np.int64)
    si = np.asarray(pc.index_in(syms, value_set=u_syms).to_numpy(zero_copy_only=False), dtype=np.int64)
    cols, names = [u_dates], ["date"]
    value_cols = [c for c in long_table.column_names if c not in (date_col, symbol_col)]
    for k, sym in enumerate(u_syms.to_pylist()):
        rows = np.nonzero(si == k)[0]
        where = np.full(len(u_dates), -1, dtype=np.int64)
        where[di[rows]] = rows
        take = pa.array(where, mask=where < 0)
        for c in value_cols:
            cols.append(long_table[c].combine_chunks().take(take))
            names.append("%s_%s" % (sym, c))
    return pa.table(cols, names=names)


def split_columns(table: pa.Table, fields):
    """-> (symbols in order of first appearance, {field: {symbol: column name}}) for `{symbol}_{field}` columns."""
    symbols, by_field = {}, {f: {} for f in fields}
    for name in table.column_names:
        sym, sep, f = name.rpartition("_")
        if sep and sym and f in by_field:
            by_field[f][sym] = name
            symbols.setdefault(sym, None)
    return list(symbols), by_field


_extra_engines: dict[tuple[int, int], Engine] = {}      # (device, k) -> the k-th further engine of a device (k >= 1)


def _shard_engines(devices) -> list[Engine]:
    """One engine per entry of `devices`.  A panel run drives its engine's streams and fork / join events (include/pqb200.h:
    one engine per thread), so shards that share a device must not share an engine: the first occurrence of an ordinal
    gets `get_engine(d)`, every repeat a further engine of that device, created once and reused by later calls."""
    seen: dict[int, int] = {}
    out = []
    for d in devices:
        k = seen[d] = seen.get(d, -1) + 1
        if k == 0:
            out.append(get_engine(d))
            continue
        if (d, k) not in _extra_engines:
            _extra_engines[(d, k)] = Engine(d)
        out.append(_extra_engines[(d, k)])
    return out


def _f64(col) -> pa.Array:
    a = col.combine_chunks() if isinstance(col, pa.ChunkedArray) else col
    return a if a.type == pa.float64() else a.cast(pa.float64())


def _set(setter, handle, symbol, field, arr: pa.Array, n):
    bufs = arr.buffers()
    vptr = C.c_void_p(bufs[0].address) if (bufs[0] is not None and arr.null_count) else None
    N.check(setter(handle, symbol, field, C.c_void_p(bufs[1].address), vptr, arr.offset, n))


class _Keep:
    """Base object of the zero-copy result buffers: keeps the panel (its pinned memory) alive."""

    def __init__(self, owner):
        self.owner = owner


class WideResult:
    """The result of `WidePanel.suite(lazy=True)`: the `{symbol}_{output}` columns of a run, made on demand as Arrow arrays
    that alias the pinned result planes (no copy; an array keeps its panel alive).  A 2,000-symbol suite has 42,000 result
    columns: wrapping every one of them in Arrow objects costs more host time than the GPU pass (pyarrow needs ~1 us per
    column and per operation), so the wide table is only built when `table()` is called.

        res = wp.suite(lazy=True)
        res["AAPL_rsi"]            # pyarrow Float64 array (values + validity straight from the pinned planes)
        res.symbol("AAPL")         # {"sma": array, "ema": array, ...}
        res.matrix("rsi")          # (values [n_symbols, n_bars] numpy view, validity bool [n_symbols, n_bars])
        res.table()                # the full `date` + `{symbol}_{output}` pyarrow table"""

    def __init__(self, shards, symbols, names, omask, n_bars, dates):
        self._shards = shards                  # [(Panel, lo, hi)]
        # (columns in the order of the table: by symbol, then by output id)
        self.symbols, self.outputs = list(symbols), sorted(names, key=N.OUTPUT_NAMES.index)
        self._omask, self.n_bars, self.dates = omask, n_bars, dates
        self._row = {s: i for i, s in enumerate(self.symbols)}
        self._by_len = sorted(self.outputs, key=len, reverse=True)

    def __len__(self):
        return len(self.symbols) * len(self.outputs)

    @property
    def column_names(self):
        return ["%s_%s" % (s, o) for s in self.symbols for o in self.outputs]

    def _locate(self, row):
        for p, lo, hi in self._shards:
            if lo <= row < hi:
                return p, row - lo
        raise KeyError(row)

    def array(self, symbol: str, output: str) -> pa.Array:
        p, r = self._locate(self._row[symbol])
        k = N.OUTPUT_NAMES.index(output)
        if output not in self.outputs:
            raise KeyError(output)
        base = _Keep(p)
        vals = N.lib().pqb_panel_host_output(p._h, k) + r * p.pitch * 8
        bits = N.lib().pqb_panel_host_validity(p._h, k) + r * p.validity_pitch
        return pa.Array.from_buffers(pa.float64(), self.n_bars, [pa.foreign_buffer(bits, (self.n_bars + 7) // 8, base),
                                                                 pa.foreign_buffer(vals, self.n_bars * 8, base)])

    def __getitem__(self, name: str) -> pa.Array:
        for o in self._by_len:                 # `{symbol}_{output}`: symbols may contain underscores themselves
            if name.endswith("_" + o) and name[:-len(o) - 1] in self._row:
                return self.array(name[:-len(o) - 1], o)
        raise KeyError(name)

    def symbol(self, symbol: str) -> dict:
        return {o: self.array(symbol, o) for o in self.outputs}

    def matrix(self, output: str):
        """(values, validity) of one output for every symbol, rows in `symbols` order (numpy; one shard: views)."""
        k = N.OUTPUT_NAMES.index(output)
        vs = [p.host_output(k) for p, _, _ in self._shards]
        oks = [p.host_validity(k) for p, _, _ in self._shards]
        return (vs[0], oks[0]) if len(vs) == 1 else (np.concatenate(vs), np.concatenate(oks))

    def table(self) -> pa.Table:
        batches = [p.export_arrow(self._omask, self.symbols[lo:hi]) for p, lo, hi in self._shards]
        if len(batches) == 1:
            out = pa.Table.from_batches(batches)
        else:
            cols, names = [], []
            for rb in batches:
                cols.extend(rb.columns)
                names.extend(rb.schema.names)
            out = pa.table(cols, names=names)
        if self.dates is not None:
            out = out.add_column(0, "date", self.dates)
        return out


class WidePanel:
    """A wide `date` + `{symbol}_{column}` table on one B200."""

    def __init__(self, table: pa.Table, engine: Engine | None = None):
        self.table = table
        self.engine = engine
        self.dates = table["date"] if "date" in table.column_names else None
        self.n_bars = table.num_rows
        self._index = {name: i for i, name in enumerate(table.column_names)}     # (Table[name] is slow on wide tables)
        self._suite = None
        self._candles = None
        self._batch = None
        self._exported = None
        self.last_timings = {}

    def _col(self, name):
        return self.table.column(self._index[name])

    # ---- the 15-indicator suite (+ optional groups through `params.indicators`) ----
    def _suite_map(self, symbols, cols):
        """column index -> (symbol row, field) arrays for pqb_*_record_batch (field -1: not a panel column)."""
        sym = np.zeros(self.table.num_columns, dtype=np.int64)
        fld = np.full(self.table.num_columns, -1, dtype=np.int32)
        for f, fname in enumerate(SUITE_FIELDS):
            by = cols[fname]
            idx = np.fromiter((self._index[by[s]] for s in symbols), dtype=np.int64, count=len(symbols))
            sym[idx] = np.arange(len(symbols))
            fld[idx] = f
        return sym, fld

    def _record_batch(self):
        """The table as ONE record batch exported through the Arrow C Data Interface (zero copy for a single-chunk table)."""
        if self._batch is None:
            t = self.table if all(c.num_chunks <= 1 for c in self.table.columns) else self.table.combine_chunks()
            batches = t.to_batches()
            self._batch = batches[0] if batches else pa.RecordBatch.from_pylist([], schema=t.schema)
        arr, sch = N.ArrowArray(), N.ArrowSchema()
        self._batch._export_to_c(C.addressof(arr), C.addressof(sch))
        return arr, sch

    def _record_batch_cached(self):
        """One export for the life of this WidePanel (the table is immutable): exporting 10,001 columns through the C Data
        Interface costs ~5 ms per call.  The engine only borrows the batch (it never calls release)."""
        if self._exported is None:
            self._exported = self._record_batch()
        return self._exported

    def __del__(self):
        try:
            if self._exported is not None:
                self._release(*self._exported)
                self._exported = None
        except Exception:
            pass

    @staticmethod
    def _release(arr, sch):
        for x, proto in ((arr, C.CFUNCTYPE(None, C.POINTER(N.ArrowArray))), (sch, C.CFUNCTYPE(None, C.POINTER(N.ArrowSchema)))):
            if x.release:
                proto(x.release)(C.pointer(x))

    def suite(self, params: N.SuiteParams | None = None, outputs=None, threads: int = 0, devices=None, lazy: bool = False):
        """Runs the fused suite over every symbol that has close / high / low / volume columns; returns `date` +
        `{symbol}_{output}` for the requested output names (default: the 21 suite outputs).  The table crosses the C ABI
        as ONE Arrow record batch (pqb_suite_run_record_batch: intake pipelined with the GPU pipeline) and the results
        come back as ONE record batch aliasing the pinned result planes (pqb_panel_export_arrow) -- no per-column work in
        Python.  `devices`: GPU ordinals to shard the symbols over (contiguous ranges, one host thread per GPU, no
        collective -- SURVEY.md 8e); default: this panel's engine only.  Every shard runs on an engine of its own: an
        ordinal listed more than once (e.g. `[0, 0]`, several shards on one GPU) gets a further engine of that device per
        repeat, kept for later calls.  `lazy=True` returns a `WideResult` (columns wrapped on demand) instead of the full
        table."""
        import time
        tm = self.last_timings = {}
        t_ = time.perf_counter()

        def lap(name):
            nonlocal t_
            now = time.perf_counter()
            tm[name] = tm.get(name, 0.0) + (now - t_) * 1e3
            t_ = now

        symbols, cols = split_columns(self.table, SUITE_FIELDS)
        symbols = [s for s in symbols if all(s in cols[f] for f in SUITE_FIELDS)]
        if not symbols:
            raise ValueError("no symbol has all of " + ", ".join("{symbol}_" + f for f in SUITE_FIELDS))
        params = params or N.default_params()
        names = list(outputs) if outputs is not None else N.OUTPUT_NAMES[:N.N_SUITE_OUTPUTS]
        omask = sum(1 << N.OUTPUT_NAMES.index(n) for n in names)
        self._suite = None          # (an earlier panel no result refers to any more goes back to the engine's pinned pool first)
        lap("release_previous_panel_ms")
        sym, fld = self._suite_map(symbols, cols)
        lap("column_map_ms")
        engines = [self.engine or get_engine(0)] if not devices else _shard_engines(devices)
        from .shard import symbol_range
        shards = []
        for g, eng in enumerate(engines):
            lo, hi = symbol_range(len(symbols), len(engines), g)
            if hi > lo:
                shards.append((eng, lo, hi))
        batches = [None] * len(shards)
        errors = []

        def run(i):
            eng, lo, hi = shards[i]
            try:
                t0 = time.perf_counter()
                p = Panel(hi - lo, self.n_bars, engine=eng, outputs_mask=omask, host_staging=2)     # (every row is staged below)
                tm["panel_create_ms"] = tm.get("panel_create_ms", 0.0) + (time.perf_counter() - t0) * 1e3
                mine = (fld >= 0) & (sym >= lo) & (sym < hi)
                s_i = np.ascontiguousarray(np.where(mine, sym - lo, 0), dtype=np.int64)
                f_i = np.ascontiguousarray(np.where(mine, fld, -1), dtype=np.int32)
                t0 = time.perf_counter()
                arr, sch = self._record_batch_cached()
                t1 = time.perf_counter()
                N.check(N.lib().pqb_suite_run_record_batch(p._h, C.byref(params), C.byref(arr), C.byref(sch), s_i.ctypes.data,
                                                           f_i.ctypes.data, threads))
                t2 = time.perf_counter()
                batches[i] = (p, None if lazy else p.export_arrow(omask, symbols[lo:hi]))
                t3 = time.perf_counter()
                for k, v in (("export_input_batch_ms", t1 - t0), ("run_record_batch_ms", t2 - t1), ("export_results_ms", t3 - t2)):
                    tm[k] = tm.get(k, 0.0) + v * 1e3
            except Exception as ex:                      # (raised again on the calling thread)
                errors.append(ex)

        if len(shards) == 1:
            run(0)
        else:
            import threading
            ts = [threading.Thread(target=run, args=(i,)) for i in range(len(shards))]
            for t in ts:
                t.start()
            for t in ts:
                t.join()
        if errors:
            raise errors[0]
        t_ = time.perf_counter()
        self._suite = [p for p, _ in batches]
        if lazy:
            res = WideResult([(b[0], sh[1], sh[2]) for b, sh in zip(batches, shards)], symbols, names, omask, self.n_bars, self.dates)
            lap("assemble_table_ms")
            return res
        if len(batches) == 1:
            out = pa.Table.from_batches([batches[0][1]])
        else:
            out_cols, out_names = [], []
            for _, rb in batches:
                out_cols.extend(rb.columns)
                out_names.extend(rb.schema.names)
            out = pa.table(out_cols, names=out_names)
        if self.dates is not None:
            out = out.add_column(0, "date", self.dates)
        lap("assemble_table_ms")
        return out

    # ---- live: append new rows to the computed table ----
    def live(self, params: N.SuiteParams | None = None, outputs=None, max_push_bars: int = 64, devices=None,
             nulls: bool = False, screen=None) -> "WideLive":
        """A live panel primed from this table (include/pqb200.h "live panels"): `.push(rows)` takes k new rows in the
        table's own `date` + `{symbol}_{field}` shape and returns `date` + `{symbol}_{output}` for those rows -- the
        columns, names and values `suite()` of the concatenated table gives for them.  One GPU (`devices` is refused).
        nulls=True: the table and the pushed rows may have halted cells; after each push `WideLive.voided` lists the
        `{symbol}_{output}` columns whose earlier rows that push turned null.  screen (see LivePanel): after each push
        `WideLive.signals` holds `date` + `{symbol}_{signal}` Int8 columns, and `WideLive.info()` equals `info()` of the
        concatenated table."""
        if devices:
            raise NotImplementedError("live panels run on one GPU: multi-GPU live panels are not built")
        symbols, cols = split_columns(self.table, SUITE_FIELDS)
        symbols = [s for s in symbols if all(s in cols[f] for f in SUITE_FIELDS)]
        if not symbols:
            raise ValueError("no symbol has all of " + ", ".join("{symbol}_" + f for f in SUITE_FIELDS))
        params = params or N.default_params()
        names = list(outputs) if outputs is not None else N.OUTPUT_NAMES[:N.N_SUITE_OUTPUTS]
        omask = sum(1 << N.OUTPUT_NAMES.index(n) for n in names)
        sym, fld = self._suite_map(symbols, cols)
        p = Panel(len(symbols), self.n_bars, engine=self.engine or get_engine(0), outputs_mask=0, host_staging=2)
        try:
            arr, sch = self._record_batch_cached()
            N.check(N.lib().pqb_panel_set_record_batch(p._h, C.byref(arr), C.byref(sch), sym.ctypes.data, fld.ctypes.data, 0))
            p.upload()
            from .live import LivePanel
            lp = LivePanel(p, params, omask, max_push_bars, nulls=nulls, screen=screen)
        finally:
            p.close()
        wl = WideLive(lp, symbols, {f: cols[f] for f in SUITE_FIELDS}, sorted(names, key=N.OUTPUT_NAMES.index))
        if lp.screen is not None and lp.screen.info:
            # info() lists symbols in the order of the table's close / high / low / volume / open columns
            info_syms, ocols = split_columns(self.table, SUITE_FIELDS + ("open",))
            wl._info_order = [symbols.index(s) for s in info_syms if s in wl._index]
            wl._open_cols = ocols["open"]
            last = self.n_bars - 1
            wl._open = [self._col(ocols["open"][s])[last].as_py() if s in ocols["open"] else None for s in symbols]
        return wl

    # ---- Selector.info(): last-row reductions (README.md:832-851) ----
    def info(self) -> pa.Table:
        """One row per symbol with the README's 15 `Selector.info()` columns: symbol, price, open, high, low, volume,
        return_1d / 5d / 20d, volatility, ma_5 / 10 / 20, volume_ratio, amplitude (arithmetic: include/pqb200.h
        `pqb_panel_info`).  `open` is the last row of `{symbol}_open` (null when the table has no such column)."""
        symbols, cols = split_columns(self.table, SUITE_FIELDS + ("open",))
        symbols = [s for s in symbols if all(s in cols[f] for f in SUITE_FIELDS)]
        if not symbols:
            raise ValueError("no symbol has all of " + ", ".join("{symbol}_" + f for f in SUITE_FIELDS))
        p = Panel(len(symbols), self.n_bars, engine=self.engine, outputs_mask=1)
        sym_i, fld_i = self._suite_map(symbols, cols)
        arr, sch = self._record_batch()
        try:
            N.check(N.lib().pqb_panel_set_record_batch(p._h, C.byref(arr), C.byref(sch), sym_i.ctypes.data, fld_i.ctypes.data, 0))
        finally:
            self._release(arr, sch)
        p.upload()
        res = p.info()
        last = self.n_bars - 1
        opens = [self._col(cols["open"][s])[last].as_py() if s in cols["open"] else None for s in symbols]
        out = {"symbol": pa.array(symbols), "price": None, "open": pa.array(opens, type=pa.float64())}
        for name in N.INFO_NAMES:
            v, ok = res[name]
            out[name] = pa.array(v, mask=~ok)
        order = ["symbol", "price", "open", "high", "low", "volume", "return_1d", "return_5d", "return_20d", "volatility",
                 "ma_5", "ma_10", "ma_20", "volume_ratio", "amplitude"]
        return pa.table([out[n] for n in order], names=order)

    # ---- candles: 61 cdl* patterns + price transforms + bop ----
    def candles(self, params: N.CandleParams | None = None, patterns=None, prices=None, on_nulls: str = "error") -> pa.Table:
        """`date` + `{symbol}_{cdl*}` (Int32) + `{symbol}_{avgprice,...,bop}`.  The reference's cdl* and bop fail on a
        column with nulls (`cont_slice()?`): `on_nulls="error"` raises naming the symbols, `"skip"` leaves them out."""
        symbols, cols = split_columns(self.table, CANDLE_FIELDS)
        symbols = [s for s in symbols if all(s in cols[f] for f in CANDLE_FIELDS)]
        if not symbols:
            raise ValueError("no symbol has all of " + ", ".join("{symbol}_" + f for f in CANDLE_FIELDS))
        with_nulls = [s for s in symbols if any(self._col(cols[f][s]).null_count for f in CANDLE_FIELDS)]
        if with_nulls:
            if on_nulls != "skip":
                raise ValueError("open/high/low/close of %s have nulls: the reference's cdl* / bop refuse such columns "
                                 "(cont_slice()?); pass on_nulls='skip' to leave them out" % ", ".join(with_nulls[:8]))
            symbols = [s for s in symbols if s not in with_nulls]
            if not symbols:
                raise ValueError("every symbol has nulls in open/high/low/close")
        all_names = pattern_names()
        pat = list(patterns) if patterns is not None else all_names
        prc = list(prices) if prices is not None else list(N.PRICE_NAMES)
        pmask = sum(1 << all_names.index(n) for n in pat)
        rmask = sum(1 << N.PRICE_NAMES.index(n) for n in prc)
        cp = CandlePanel(len(symbols), self.n_bars, engine=self.engine, patterns_mask=pmask, prices_mask=rmask)
        for s, sym in enumerate(symbols):
            for f, fname in enumerate(CANDLE_FIELDS):
                arr = _f64(self._col(cols[fname][sym]))
                _set(N.lib().pqb_candles_set_column, cp._h, s, f, arr, self.n_bars)
        prm = params or candle_default_params(pmask, rmask)
        prm.patterns, prm.prices = pmask, rmask
        cp.run_host(prm)
        self._candles = cp
        base = _Keep(cp)
        out_cols, out_names = ([self.dates], ["date"]) if self.dates is not None else ([], [])
        vbytes = (self.n_bars + 7) // 8
        for s, sym in enumerate(symbols):
            for n in pat:
                ptr = N.lib().pqb_candles_host_pattern(cp._h, all_names.index(n)) + s * cp.pitch * 4
                out_cols.append(pa.Array.from_buffers(pa.int32(), self.n_bars, [None, pa.foreign_buffer(ptr, self.n_bars * 4, base)]))
                out_names.append("%s_%s" % (sym, n))
            for n in prc:
                k = N.PRICE_NAMES.index(n)
                vals = N.lib().pqb_candles_host_price(cp._h, k) + s * cp.pitch * 8
                bits = N.lib().pqb_candles_host_price_validity(cp._h, k) + s * cp.words_per_row * 4
                out_cols.append(pa.Array.from_buffers(pa.float64(), self.n_bars,
                                                      [pa.foreign_buffer(bits, vbytes, base), pa.foreign_buffer(vals, self.n_bars * 8, base)]))
                out_names.append("%s_%s" % (sym, n))
        return pa.table(out_cols, names=out_names)


class WideLive:
    """`WidePanel.live()`: pushes k new rows of the wide table, returns their `date` + `{symbol}_{output}` rows."""

    def __init__(self, live, symbols, cols, outputs):
        self.live, self.symbols, self._cols, self.outputs = live, symbols, cols, outputs
        self.voided: list[str] = []             # `{symbol}_{output}` columns whose earlier rows the last push made null
        self.signals: pa.Table | None = None    # screen: `date` + `{symbol}_{signal}` of the last push
        self._index = {s: j for j, s in enumerate(symbols)}
        self._info_order, self._open_cols, self._open = None, {}, []

    @property
    def bars(self) -> int:
        return self.live.bars

    def push(self, rows: pa.Table, commit: bool = True) -> pa.Table:
        k = rows.num_rows
        vals, valid = {}, {}
        index = {name: i for i, name in enumerate(rows.column_names)}
        for f in SUITE_FIELDS:
            v = np.empty((k, len(self.symbols)), dtype=np.float64)
            ok = np.empty((k, len(self.symbols)), dtype=bool)
            for j, s in enumerate(self.symbols):
                a = _f64(rows.column(index[self._cols[f][s]]))
                ok[:, j] = ~np.asarray(a.is_null(), dtype=bool) if a.null_count else True
                v[:, j] = a.to_numpy(zero_copy_only=False)
            vals[f], valid[f] = v, ok
        res = self.live.push(vals["close"], vals["high"], vals["low"], vals["volume"], valid=valid, commit=commit)
        self.voided = ["%s_%s" % (self.symbols[j], o) for o in self.outputs for j in self.live.voided.get(o, ())]
        out_cols, out_names = [], []
        for j, s in enumerate(self.symbols):
            for o in self.outputs:
                v, ok = res[o]
                out_cols.append(pa.array(v[j], type=pa.float64(), mask=~ok[j]))
                out_names.append("%s_%s" % (s, o))
        out = pa.table(out_cols, names=out_names)
        if "date" in index:
            out = out.add_column(0, "date", rows.column(index["date"]))
        if self.live.screen is not None:
            sig_cols, sig_names = [], []
            for j, s in enumerate(self.symbols):
                for name, a in self.live.signals.items():
                    sig_cols.append(pa.array(a[j], type=pa.int8()))
                    sig_names.append("%s_%s" % (s, name))
            self.signals = pa.table(sig_cols, names=sig_names)
            if "date" in index:
                self.signals = self.signals.add_column(0, "date", rows.column(index["date"]))
            if commit and self._info_order is not None:
                self._open = [rows.column(index[self._open_cols[s]])[k - 1].as_py() if self._open_cols.get(s) in index else None
                              for s in self.symbols]
        return out

    def info(self) -> pa.Table:
        """`WidePanel.info()` of the table with every committed push appended: one row per symbol, the README's 15
        `Selector.info()` columns (`open` from the last committed row's `{symbol}_open`, null when it has none).  Needs a
        screen with info."""
        if self._info_order is None:
            raise ValueError("info() needs a live table created with screen info (screen=True or dict(info=True))")
        res = self.live.info()
        order = self._info_order
        out = {"symbol": pa.array([self.symbols[j] for j in order]),
               "open": pa.array([self._open[j] for j in order], type=pa.float64())}
        for name in N.INFO_NAMES:
            v, ok = res[name]
            out[name] = pa.array(v[order], mask=~ok[order])
        names = ["symbol", "price", "open", "high", "low", "volume", "return_1d", "return_5d", "return_20d", "volatility",
                 "ma_5", "ma_10", "ma_20", "volume_ratio", "amplitude"]
        return pa.table([out[n] for n in names], names=names)
