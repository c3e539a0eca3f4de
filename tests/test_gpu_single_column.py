"""The single-column boundary -- the C ABI entry points (`pqb_sma`, `pqb_atr`, `pqb_stochf`, ...: `run_single` in
engine.cu) and the polars plugin symbols behind them -- against the oracle, bit for bit in values and validity, at the
shapes where its host paths part ways:

  * both staging paths: columns of up to PQB_SINGLE_MAPPED bars (default 32,768) go through the mapped pack / unpack
    kernels, longer ones through the copy engine (d_xin / d_xout, prepare_nulls); 32,768 and 32,769 sit on the two
    sides of the default, 131,073 is past the length whose scratch panel is parked, ~1 M bars is the README's example;
  * the engine's scratch-panel cache (one current panel + an LRU of 3, panels over 131,072 bars destroyed), whose
    recycled panels keep device planes, null state and validity of earlier calls;
  * Arrow validity at bit offsets that are not a multiple of 8 (copy_bits' shifting branch), chunked and cast inputs,
    through the plugin's zero-copy path and the record-batch intake;
  * the composed shims (STOCH with smoothing types, STOCHF, STOCHRSI, MACDEXT and its col_sub kernel's tail byte);
  * many threads on one engine across both staging paths.

Where the reference fails, the product must fail the same way: PQB_ERR_NULLS from the C ABI, PluginError "not
contiguous" from the plugin, PQB_ERR_UNSUPPORTED for the moving-average types that are not built (2, 3, 6, 8)."""
import ctypes as C
import threading

import numpy as np
import pyarrow as pa
import pytest

import synth
import tolerances as T
from oracle import pqo

pytestmark = pytest.mark.gpu

ERR_UNSUPPORTED, ERR_NULLS = -4, -5
LENGTHS = [1, 7, 8, 33, 252, 32_767, 32_768, 32_769, 131_073]


@pytest.fixture(scope="module")
def pq():
    import polars_quant_b200 as m
    return m


@pytest.fixture(scope="module")
def eng(pq):
    e = pq.Engine(0)
    yield e
    e.close()


def _L():
    from polars_quant_b200 import _native as N
    return N.lib()


# ---- calling the C ABI ------------------------------------------------------------------------------------------------
class _In:
    """One input column as a pqb_col: f64 values and an optional LSB-first bitmap, both kept alive with the struct.
    Null slots hold a value the reference never reads (NaN, an infinity or a huge number): the product must not read it."""

    def __init__(self, x, ok=None):
        from polars_quant_b200 import _native as N
        self.x = np.ascontiguousarray(x, dtype=np.float64)
        self.bits = None if ok is None else np.packbits(ok.astype(np.uint8), bitorder="little")
        self.col = N.Col(self.x.ctypes.data, None if self.bits is None else self.bits.ctypes.data, 0, len(self.x))


def _poison(x, ok, seed=0):
    """x with its null slots overwritten by values no reference computation may see."""
    if ok is None:
        return x
    x = x.copy()
    junk = np.array([np.nan, np.inf, -np.inf, 1e308, -1e308, 0.0])
    idx = np.nonzero(~ok)[0]
    x[idx] = junk[(idx + seed) % len(junk)]
    return x


def _call(eng, fname, ins, ints=(), floats=(), n_out=1, out_ok=None):
    """-> (rc, [(values, validity bool), ...]).  `out_ok` (a list of bools) selects pqb_dm's outputs (NULL for the others)."""
    from polars_quant_b200 import _native as N
    n = ins[0].col.len
    vals = [np.full(max(n, 1), 7.0) for _ in range(n_out)]
    bits = [np.full((n + 7) // 8 + 1, 0xA5, np.uint8) for _ in range(n_out)]
    ocs = [N.OutCol(v.ctypes.data, b.ctypes.data) for v, b in zip(vals, bits)]
    args = [eng._h] + [C.byref(i.col) for i in ins] + [C.c_int32(int(p)) for p in ints] + [C.c_double(f) for f in floats]
    if out_ok is None:
        args += [C.byref(o) for o in ocs]
    else:
        it = iter(ocs)
        args += [C.byref(next(it)) if want else None for want in out_ok]
    rc = getattr(_L(), fname)(*args)
    return rc, [(v[:n], np.unpackbits(b, bitorder="little")[:n].astype(bool)) for v, b in zip(vals, bits)]


def _same(what, got, ref):
    ref = ref if isinstance(ref, tuple) and isinstance(ref[0], tuple) else (ref,)
    assert len(got) == len(ref), what
    for j, ((gv, gk), (rv, rk)) in enumerate(zip(got, ref)):
        nbad, msg = T.compare(f"{what} out {j}", gv, gk, rv, rk)
        assert nbad == 0, msg


def _kdj_ref(h, l, c, fk, k, d, hok=None, lok=None, cok=None):
    sk, sd = pqo.stoch(h, l, c, fk, k, 0, d, 0, hok, lok, cok)
    jok = sk[1] & sd[1]
    return sk, sd, (np.where(jok, 3.0 * sk[0] - 2.0 * sd[0], np.nan), jok)


# Every single-column entry point: (C function, inputs from "chlv", period -> (ints, floats), default period, n_out,
# oracle(cols, oks, ints) with oks[i] None for a null-free input, skips nulls like the reference?)
def _entries():
    E = []

    def add(name, fn, ins, mk, dflt, n_out, ref, shift):
        E.append(dict(name=name, fn=fn, ins=ins, mk=mk, dflt=dflt, n_out=n_out, ref=ref, shift=shift))

    one = lambda p: ((p,), ())
    for nm in ("sma", "ema", "tema", "trima"):
        add(nm, "pqb_" + nm, "c", one, 30, 1, lambda X, K, P, f=getattr(pqo, nm): f(X[0], P[0], K[0]), True)
    for m in (0, 1, 4, 5, 7):
        add(f"ma{m}", "pqb_ma", "c", lambda p, m=m: ((p, m), ()), 30, 1, lambda X, K, P: pqo.ma(X[0], P[0], P[1], K[0]), True)
    add("bbands", "pqb_bbands", "c", lambda p: ((p,), (1.5, 2.5)), 20, 3, lambda X, K, P: pqo.bbands(X[0], P[0], 1.5, 2.5, K[0]), True)
    add("midpoint", "pqb_midpoint", "c", one, 14, 1, lambda X, K, P: pqo.midpoint(X[0], P[0], K[0]), True)
    add("midprice", "pqb_midprice", "hl", one, 14, 1, lambda X, K, P: pqo.midprice(X[0], X[1], P[0], K[0], K[1]), False)
    add("trange", "pqb_trange", "hlc", lambda p: ((), ()), 0, 1, lambda X, K, P: pqo.trange(*X, *K), True)
    add("atr", "pqb_atr", "hlc", one, 14, 1, lambda X, K, P: pqo.atr(*X, P[0], *K), True)
    add("natr", "pqb_natr", "hlc", one, 14, 1, lambda X, K, P: pqo.natr(*X, P[0], *K), True)
    add("obv", "pqb_obv", "cv", lambda p: ((), ()), 0, 1, lambda X, K, P: pqo.obv(*X, *K), True)
    add("ad", "pqb_ad", "hlcv", lambda p: ((), ()), 0, 1, lambda X, K, P: pqo.ad(*X, *K), True)
    add("adosc", "pqb_adosc", "hlcv", lambda p: ((3, 10) if p is None else (p, p), ()), None, 1,
        lambda X, K, P: pqo.adosc(*X, P[0], P[1], *K), True)
    add("willr", "pqb_willr", "hlc", one, 14, 1, lambda X, K, P: pqo.willr(*X, P[0], *K), False)
    add("rsi", "pqb_rsi", "c", one, 14, 1, lambda X, K, P: pqo.rsi(X[0], P[0], K[0]), False)
    add("macd", "pqb_macd", "c", lambda p: ((12, 26, 9) if p is None else (p, p, p), ()), None, 3,
        lambda X, K, P: pqo.macd(X[0], *P, ok=K[0]), False)
    add("kdj", "pqb_kdj", "hlc", lambda p: ((9, 3, 3) if p is None else (p, p, p), ()), None, 3,
        lambda X, K, P: _kdj_ref(*X, *P, *K), True)
    add("stoch", "pqb_stoch", "hlc", lambda p: ((5, 3, 3) if p is None else (p, p, p), ()), None, 2,
        lambda X, K, P: pqo.stoch(*X, P[0], P[1], 0, P[2], 0, *K), True)
    add("mom", "pqb_mom", "c", one, 10, 1, lambda X, K, P: pqo.mom(X[0], P[0], K[0]), False)
    for kind in range(4):
        add(f"roc{kind}", "pqb_roc", "c", lambda p, k=kind: ((p, k), ()), 10, 1, lambda X, K, P: pqo.roc(X[0], P[0], P[1], K[0]), False)
    add("cmo", "pqb_cmo", "c", one, 14, 1, lambda X, K, P: pqo.cmo(X[0], P[0], K[0]), False)
    add("mfi", "pqb_mfi", "hlcv", one, 14, 1, lambda X, K, P: pqo.mfi(*X, P[0]), False)
    add("cci", "pqb_cci", "hlc", one, 14, 1, lambda X, K, P: pqo.cci(*X, P[0], *K), False)
    add("trix", "pqb_trix", "c", one, 30, 1, lambda X, K, P: pqo.trix(X[0], P[0], K[0]), False)
    add("ultosc", "pqb_ultosc", "hlc", lambda p: ((7, 14, 28) if p is None else (p, p, p), ()), None, 1,
        lambda X, K, P: pqo.ultosc(*X, *P), False)
    add("aroon", "pqb_aroon", "hl", one, 14, 2, lambda X, K, P: pqo.aroon(X[0], X[1], P[0]), False)
    add("donchian", "pqb_donchian", "hl", one, 20, 2, lambda X, K, P: pqo.donchian(X[0], X[1], P[0]), False)
    add("dm", "pqb_dm", "hlc", one, 14, 6, lambda X, K, P: tuple(pqo.dm(*X, P[0]).values()), False)
    return E


ENTRIES = _entries()
_FIELD = {"c": "close", "h": "high", "l": "low", "v": "volume"}


def _null_patterns(n, seed):
    """name -> validity (bool[n]) of the null patterns a real column has."""
    rng = np.random.default_rng(seed)
    pats = {}
    ok = np.ones(n, bool); ok[:max(1, n // 3)] = False; pats["late listing"] = ok
    ok = np.ones(n, bool); ok[7:9] = False; ok[31:34] = False; ok[n // 2:n // 2 + 3] = False; pats["halts 7-8, 31-33"] = ok
    ok = np.ones(n, bool); ok[8:32] = False; ok[33:34] = False; pats["halts 8-31, 33"] = ok
    ok = np.ones(n, bool); ok[n - max(1, n // 4):] = False; pats["delisting"] = ok
    ok = np.zeros(n, bool); ok[n // 2] = True; pats["one valid bar"] = ok
    pats["all null"] = np.zeros(n, bool)
    ok = rng.random(n) > 0.05; ok[:5] = False; pats["scattered"] = ok
    return pats


def _one_input(e):
    """The input that carries nulls alone in the 'nulls in one input only' case."""
    return {"obv": "v", "ad": "v", "adosc": "v"}.get(e["name"], "h" if "h" in e["ins"] else None)


_ORACLE_WITHOUT_VALIDITY = ("mfi", "ultosc", "aroon", "donchian", "dm")


def _refused_long_window(rc, ints, n, where):
    """A window of more than 128 bars, longer than the column, whose per-block rings do not fit one launch's shared memory
    (KDJ's three windows of 253 bars already need 299,584 bytes) is refused loudly with PQB_ERR_UNSUPPORTED (include/pqb200.h:
    "valid in the reference but outside this build"), never answered with a wrong column.  True when that is what happened;
    shorter windows must run."""
    if rc != ERR_UNSUPPORTED or max(ints, default=0) <= max(n, 128):
        return False
    assert "shared memory" in _L().pqb_last_error().decode(), where
    return True


def _all_of(cases):
    """Runs every case (a callable that asserts) and reports every mismatch at once, not just the first."""
    fails = []
    for where, fn in cases:
        try:
            fn()
        except AssertionError as ex:
            fails.append(f"{where}: {str(ex).splitlines()[0]}")
    assert not fails, f"{len(fails)} mismatches:\n" + "\n".join(fails[:40])


def _run_entry(eng, e, d, oks, P, where):
    """One call of entry `e` against the oracle on the same inputs: bit-exact, or the reference's failure."""
    cols = [d[_FIELD[f]] for f in e["ins"]]
    ks = [oks.get(f) for f in e["ins"]]
    ints, floats = P
    ins = [_In(_poison(x, k, j), k) for j, (x, k) in enumerate(zip(cols, ks))]
    any_null = any(k is not None and not k.all() for k in ks)
    rc, got = _call(eng, e["fn"], ins, ints, floats, e["n_out"])
    if any_null and not e["shift"]:
        # momentum.rs functions (and midprice) fail on a column with nulls in the reference (cont_slice()?)
        assert rc == ERR_NULLS, f"{where}: rc {rc}, expected PQB_ERR_NULLS"
        if e["name"] in _ORACLE_WITHOUT_VALIDITY:
            return
        if e["name"] == "midprice" and ks[1] is None:
            # nulls in high alone: the reference computes, the engine refuses (it would need the high pass's own start:
            # engine.cu pqb_midprice) -- a documented refusal, never a wrong column
            return
        with pytest.raises(pqo.OracleError):
            e["ref"](cols, ks, ints)
        return
    ref = e["ref"](cols, ks, ints)
    if _refused_long_window(rc, ints, len(cols[0]), where):
        return
    assert rc == 0, f"{where}: rc {rc}: {_L().pqb_last_error().decode()}"
    _same(where, got, ref)


def _entry_cases(n, seed):
    """(entry, validity per input, params, label) for every entry point at length n."""
    pats = _null_patterns(n, seed)
    for e in ENTRIES:
        periods = [None] if e["dflt"] == 0 else [1, e["dflt"], n + 1]          # (trange / obv / ad take no period)
        for p in periods:
            yield e, {}, e["mk"](p), f"{e['name']} n={n} period {p}"
        dp = e["mk"](e["dflt"] or None)
        if not e["shift"]:
            yield e, {f: pats["halts 7-8, 31-33"] for f in e["ins"]}, dp, f"{e['name']} n={n} with nulls"
            continue
        for pn, ok in pats.items():
            yield e, {f: ok for f in e["ins"]}, dp, f"{e['name']} n={n} nulls: {pn}"
        f1 = _one_input(e)
        if f1 is not None:
            for pn in ("late listing", "halts 7-8, 31-33", "scattered"):
                yield e, {f1: pats[pn]}, dp, f"{e['name']} n={n} nulls in {_FIELD[f1]} only: {pn}"
    # midprice accepts no null in high either (documented refusal), and fails on any null in low like the reference
    mp = next(e for e in ENTRIES if e["name"] == "midprice")
    yield mp, {"h": pats["halts 7-8, 31-33"]}, mp["mk"](14), f"midprice n={n} nulls in high only"
    yield mp, {"l": pats["late listing"]}, mp["mk"](14), f"midprice n={n} nulls in low only"


@pytest.mark.parametrize("n", LENGTHS)
def test_every_entry_point_on_both_staging_paths(eng, n):
    """Every single-column entry point at lengths on both sides of the mapped / copy-engine threshold, periods 1, the
    default and one longer than the column, and every null pattern of a real column for the functions that skip nulls."""
    d = {k: v[0] for k, v in synth.ohlcv(1, n, seed=5000 + n).items()}
    _all_of((where, lambda e=e, oks=oks, P=P, where=where: _run_entry(eng, e, d, oks, P, where))
            for e, oks, P, where in _entry_cases(n, seed=n))


def test_a_million_bars_through_the_copy_engine(eng):
    """The README's own example of the copy-engine path: EMA, MACD, ATR and OBV over ~1 M bars, clean and with nulls."""
    n = 1_000_003
    d = {k: v[0] for k, v in synth.ohlcv(1, n, seed=77, sigma=0.0005).items()}
    pats = _null_patterns(n, seed=1)
    cases = []
    for e in ENTRIES:
        if e["name"] not in ("ema", "macd", "atr", "obv"):
            continue
        for p in ([None] if e["dflt"] == 0 else [1, e["dflt"], n + 1]):
            cases.append((e, {}, e["mk"](p), f"{e['name']} n={n} period {p}"))
        dp = e["mk"](e["dflt"] or None)
        for pn in ("late listing", "halts 7-8, 31-33", "delisting", "scattered"):
            cases.append((e, {f: pats[pn] for f in e["ins"]}, dp, f"{e['name']} n={n} nulls: {pn}"))
    _all_of((where, lambda e=e, oks=oks, P=P, where=where: _run_entry(eng, e, d, oks, P, where)) for e, oks, P, where in cases)


# ---- the scratch-panel cache ------------------------------------------------------------------------------------------
def test_recycled_scratch_panels_forget_earlier_calls(pq, eng):
    """One engine, a scripted sequence of calls: lengths cycle through more than the LRU holds (panels are parked, evicted,
    created again; 200,000 bars is destroyed instead of parked), null-bearing and clean calls alternate, and so do the
    fields each call uploads (OBV with nulls in volume then ATR, KDJ then SMA, a multi-output function then a single-output
    one), and earlier lengths come back after another function used their panel.  Every result equals the same call on a
    fresh engine and the oracle."""
    E = {e["name"]: e for e in ENTRIES}
    lens = [300, 1000, 40_000, 200_000, 64, 513, 300, 40_000, 1000, 200_000, 513, 64, 300]
    script = []
    for i, n in enumerate(lens):
        pats = _null_patterns(n, seed=i)
        halts = pats["halts 7-8, 31-33"]
        pairs = [[("obv", {"v": halts}), ("atr", {})],                                  # volume's plane, then not uploaded
                 [("kdj", {"h": halts, "l": halts, "c": halts}), ("sma", {})],           # high / low planes, then close only
                 [("bbands", {"c": pats["late listing"]}), ("ema", {})],                 # three outputs, then one
                 [("macd", {}), ("trange", {"h": pats["scattered"]})],
                 [("ad", {"v": pats["delisting"]}), ("sma", {"c": pats["one valid bar"]})],
                 [("dm", {}), ("obv", {})]]
        script += [(n, name, oks) for name, oks in pairs[(2 * i) % 6] + pairs[(2 * i + 1) % 6]]
    data = {n: {k: v[0] for k, v in synth.ohlcv(1, n, seed=n).items()} for n in set(lens)}
    for step, (n, name, oks) in enumerate(script):
        e = E[name]
        P = e["mk"](e["dflt"] or None)
        where = f"step {step}: {name} n={n} nulls in {sorted(oks)}"
        _run_entry(eng, e, data[n], oks, P, where)
        if step % 4 == 0:                                   # the same call on an engine that has seen nothing else
            fresh = pq.Engine(0)
            try:
                _run_entry(fresh, e, data[n], oks, P, where + " (fresh engine)")
            finally:
                fresh.close()


# ---- the Arrow boundary: offsets, chunks, casts ------------------------------------------------------------------------
def _arrow_np(a):
    """The combined, f64-cast column: (values with 0.0 under nulls, validity) -- what the reference computes on."""
    a = a.combine_chunks() if isinstance(a, pa.ChunkedArray) else a
    ok = ~np.asarray(a.is_null())
    v = np.asarray(a.cast(pa.float64(), safe=False).to_numpy(zero_copy_only=False), dtype=np.float64)
    return np.where(ok, v, 0.0), ok


def _plugin_same(what, got, ref):
    outs = [got.field(i) for i in range(got.type.num_fields)] if isinstance(got.type, pa.StructType) else [got]
    ref = ref if isinstance(ref[0], tuple) else (ref,)
    assert len(outs) == len(ref), what
    for j, (g, (rv, rk)) in enumerate(zip(outs, ref)):
        gok = ~np.asarray(g.is_null())
        gv = np.where(gok, np.asarray(g.to_numpy(zero_copy_only=False), dtype=np.float64), np.nan)
        nbad, msg = T.compare(f"{what} out {j}", gv, gok, rv, rk)
        assert nbad == 0, msg


# plugin function -> (inputs from "chlv", params, oracle(cols, oks))
_PLUGIN = {
    "sma": ("c", [10], lambda X, K: pqo.sma(X[0], 10, K[0])),
    "ema": ("c", [12], lambda X, K: pqo.ema(X[0], 12, K[0])),
    "tema": ("c", [5], lambda X, K: pqo.tema(X[0], 5, K[0])),
    "trima": ("c", [9], lambda X, K: pqo.trima(X[0], 9, K[0])),
    "bbands": ("c", [20, 1.5, 2.5], lambda X, K: pqo.bbands(X[0], 20, 1.5, 2.5, K[0])),
    "midpoint": ("c", [14], lambda X, K: pqo.midpoint(X[0], 14, K[0])),
    "trange": ("hlc", [], lambda X, K: pqo.trange(*X, *K)),
    "atr": ("hlc", [14], lambda X, K: pqo.atr(*X, 14, *K)),
    "natr": ("hlc", [7], lambda X, K: pqo.natr(*X, 7, *K)),
    "obv": ("cv", [], lambda X, K: pqo.obv(*X, *K)),
    "ad": ("hlcv", [], lambda X, K: pqo.ad(*X, *K)),
    "adosc": ("hlcv", [3, 10], lambda X, K: pqo.adosc(*X, 3, 10, *K)),
    "stoch": ("hlc", [5, 3, 1, 3, 4], lambda X, K: pqo.stoch(*X, 5, 3, 1, 3, 4, *K)),
    "kdj": ("hlc", [9, 3, 3], lambda X, K: _kdj_ref(*X, 9, 3, 3, *K)),
    "stochf": ("hlc", [5, 3, 5], lambda X, K: pqo.stochf(*X, 5, 3, 5, *K)),
    "macdext": ("c", [12, 4, 26, 7, 9, 1], lambda X, K: pqo.macdext(X[0], 12, 4, 26, 7, 9, 1, ok=K[0])),
}


def _plugin_check(name, arrays, where):
    from polars_quant_b200 import plugin
    ins, params, ref = _PLUGIN[name]
    X, K = zip(*(_arrow_np(a) for a in arrays))
    K = [None if k.all() else k for k in K]
    _plugin_same(where, plugin.call(name, list(arrays) + params), ref(list(X), K))


def _base(n, seed, nulls=True):
    d = {k: v[0] for k, v in synth.ohlcv(1, n, seed=seed).items()}
    rng = np.random.default_rng(seed)
    ok = {}
    for f in "chlv":
        k = rng.random(n) > 0.08
        k[:3 + seed % 5] = False                                  # listed late
        k[n // 2:n // 2 + 9] = False                              # a halt
        ok[f] = k if nulls else np.ones(n, bool)
    arr = {f: pa.array(_poison(d[_FIELD[f]], ok[f]), mask=~ok[f]) for f in "chlv"}
    return d, ok, arr


@pytest.mark.parametrize("n", [300, 40_001])
def test_plugin_sliced_columns_with_nulls_at_bit_offsets(n):
    """One Float64 chunk with nulls, sliced at offsets 1..9 and 33 (the zero-copy path: the validity reaches copy_bits at a
    bit offset); the inputs of one call at different offsets; a momentum function refuses like the reference."""
    from polars_quant_b200 import plugin
    _, _, arr = _base(n + 40, seed=n % 97)
    for off in list(range(1, 10)) + [33]:
        for name, (ins, _, _) in _PLUGIN.items():
            if n > 300 and name not in ("sma", "atr", "obv", "stochf", "macdext"):
                continue
            cols = [arr[f].slice(off + 2 * j, n) for j, f in enumerate(ins)]
            assert cols[0].offset == off and cols[0].null_count
            _plugin_check(name, cols, f"{name} n={n} offset {off}")
        with pytest.raises(plugin.PluginError, match="not contiguous"):
            plugin.call("rsi", [arr["c"].slice(off, n), 14])


@pytest.mark.parametrize("n", [300, 32_800])
def test_plugin_chunked_inputs_with_nulls(n):
    """Several chunks with nulls, each at its own non-zero offset, chunk edges inside a byte of the combined column; the
    inputs of one multi-input function chunked differently from each other."""
    from polars_quant_b200 import plugin
    _, _, arr = _base(n + 64, seed=3 + n % 11)

    def chunked(a, cuts, off):
        """chunks of `a` starting at `off`, each sliced at a different offset of its own source"""
        pieces, pos = [], off
        for w in cuts + [n - sum(cuts)]:
            pieces.append(a.slice(pos, w))
            pos += w
        return pa.chunked_array(pieces)

    layouts = [([5, 3, 11], 1), ([1, 1, 1, 6], 7), ([13], 3), ([8, 8], 2), ([31, 2, 9], 5)]
    for name, (ins, _, _) in _PLUGIN.items():
        if n > 300 and name not in ("sma", "ad", "stoch", "macdext"):
            continue
        for j0 in range(len(layouts)):
            cols = [chunked(arr[f], *layouts[(j0 + j) % len(layouts)]) for j, f in enumerate(ins)]
            _plugin_check(name, cols, f"{name} n={n} layout {j0}")
    with pytest.raises(plugin.PluginError, match="not contiguous"):
        plugin.call("macd", [chunked(arr["c"], [5, 3, 11], 1), 12, 26, 9])


@pytest.mark.parametrize("n", [300, 33_000])
def test_plugin_integer_and_float32_inputs_with_nulls(n):
    """int8 / int32 / int64 / uint64 / float32 columns with nulls whose slots hold extreme values (INT64_MIN, the largest
    uint64, NaN, +-inf): cast to Float64 like the reference, the values under nulls never read."""
    rng = np.random.default_rng(n)
    ok = rng.random(n) > 0.1
    ok[:4] = False
    ok[n - 3:] = False
    price = 50 + np.cumsum(rng.integers(-2, 3, n))
    vol = rng.integers(1, 10_000, n)

    def typed(vals, dtype, junk):
        v = vals.astype(dtype)
        v[~ok] = junk
        return pa.array(v, mask=~ok)

    cases = {
        "int8": typed(np.clip(price, -100, 100), np.int8, np.iinfo(np.int8).min),
        "int32": typed(price, np.int32, np.iinfo(np.int32).min),
        "int64": typed(price, np.int64, np.iinfo(np.int64).min),
        "uint64": typed(np.abs(price), np.uint64, np.iinfo(np.uint64).max),
        "float32": typed(price + 0.25, np.float32, np.nan),
        "float32 inf": typed(price + 0.5, np.float32, np.inf),
        "float32 -inf": typed(price - 0.5, np.float32, -np.inf),
    }
    vcol = typed(vol, np.int64, np.iinfo(np.int64).min)
    for what, col in cases.items():
        for name in ("sma", "ema", "bbands", "midpoint", "macdext"):
            _plugin_check(name, [col], f"{name} {what} n={n}")
        _plugin_check("obv", [col, vcol], f"obv {what} n={n}")
        sl = col.slice(5, n - 5)                                 # and at a bit offset
        _plugin_check("trima", [sl], f"trima {what} sliced n={n}")


def _wide_table(S, n, seed):
    """A `date` + `{symbol}_{close,high,low,volume}` table with late listings, halts, a delisting and fields that halt alone;
    volume as Int64 with INT64_MIN under its nulls."""
    d = synth.ohlcv(S, n, seed=seed)
    rng = np.random.default_rng(seed)
    F = ("close", "high", "low", "volume")
    ok = {f: np.ones((S, n), bool) for f in F}
    for s in range(S):
        if s % 3 == 1:
            for f in F: ok[f][s, :int(rng.integers(1, 40))] = False                # listed late
        if s % 4 == 2:
            a = int(rng.integers(20, n - 30))
            for f in F: ok[f][s, a:a + int(rng.integers(1, 12))] = False           # a halt
        if s % 5 == 3:
            for f in F: ok[f][s, n - int(rng.integers(1, 25)):] = False            # delisted
        if s % 6 == 4:
            ok[F[s % 4]][s, int(rng.integers(10, n - 10))] = False                 # one field halts alone
        if s % 7 == 5:
            ok["volume"][s, :9] = False                                            # volume starts later
    cols, names = [pa.array(np.arange(n, dtype=np.int64))], ["date"]
    for s in range(S):
        for f in F:
            if f == "volume":
                v = d[f][s].astype(np.int64)
                v[~ok[f][s]] = np.iinfo(np.int64).min
                d[f][s] = np.where(ok[f][s], v, 0).astype(np.float64)
            else:
                v = _poison(d[f][s], ok[f][s], s)
            cols.append(pa.array(v, mask=~ok[f][s]))
            names.append(f"s{s}_{f}")
    return pa.table(cols, names=names), d, ok


@pytest.mark.parametrize("k", [1, 3, 8])
def test_record_batch_of_a_sliced_table(k):
    """WidePanel over `table.slice(k)`: every column reaches the record-batch intake at an element offset (validity at a bit
    offset when k is not a multiple of 8), Int64 volumes with nulls are cast with their validity.  Equals the same table
    combined, cast to Float64 and rebuilt at offset 0, and the oracle for the symbols checked."""
    from test_gpu_nulls import _check_symbol_against_the_oracle
    from polars_quant_b200.wide import WidePanel
    S, n = 24, 300
    table, d, ok = _wide_table(S, n + k, seed=40 + k)
    sliced = table.slice(k)
    assert sliced.column(1).chunk(0).offset == k
    flat_cols = [pa.array(np.asarray(c.combine_chunks().cast(pa.float64(), safe=False).to_numpy(zero_copy_only=False)),
                          mask=np.asarray(c.combine_chunks().is_null()), type=pa.float64()) for c in sliced.columns[1:]]
    flat = pa.table([pa.array(np.arange(n, dtype=np.int64))] + flat_cols, names=sliced.column_names)
    assert all(c.chunk(0).offset == 0 for c in flat.columns)
    got = WidePanel(sliced).suite(lazy=True)
    ref = WidePanel(flat).suite(lazy=True)
    names = got.outputs
    res = {}
    for name in names:
        gv, gk = got.matrix(name)
        rv, rk = ref.matrix(name)
        assert np.array_equal(gk, rk), f"{name}: validity differs from the offset-0 Float64 table"
        assert T.same_bits(gv, rv).all(), f"{name}: values differ from the offset-0 Float64 table"
        res[name] = (gv.copy(), gk.copy())
    ds = {f: d[f][:, k:] for f in d}
    oks = {f: ok[f][:, k:] for f in ok}
    for s in range(S):
        _check_symbol_against_the_oracle(res, s, ds, oks, n)


# ---- the composed shims -------------------------------------------------------------------------------------------------
MATYPES = (0, 1, 4, 5, 7)
REFUSED = (2, 3, 6, 8)
SHIM_LENGTHS = [1, 5, 8, 13, 252, 32_769]


def _flat_prices(n, seed):
    """A price series with flat stretches: RSI pins to 0 / 100 / NaN there and its %K window sees a zero range."""
    d = {k: v[0] for k, v in synth.ohlcv(1, n, seed=seed).items()}
    c = d["close"].copy()
    for a in range(n // 7, n, max(1, n // 3)):
        c[a:a + max(3, n // 10)] = c[a]
    c[:min(n, 4)] = c[0]
    return c


@pytest.mark.parametrize("n", SHIM_LENGTHS)
def test_composed_shims(eng, n):
    """STOCH with every pair of smoothing types, STOCHF, STOCHRSI and MACDEXT with matypes {0, 1, 4, 5, 7}; periods 1, the
    defaults and longer than the column; clean columns, late listings, interior nulls and flat stretches.  Matypes 2, 3, 6,
    8 are refused with PQB_ERR_UNSUPPORTED."""
    d = {k: v[0] for k, v in synth.ohlcv(1, n, seed=900 + n).items()}
    h, l, c = d["high"], d["low"], d["close"]
    late = np.ones(n, bool); late[:max(1, n // 4)] = False
    holes = np.ones(n, bool); holes[3:5] = False; holes[n // 2] = False
    inputs = {"clean": {}, "late listing": {"h": late, "l": late, "c": late}, "interior nulls": {"h": holes, "l": holes, "c": holes}}
    periods = {"1": (1, 1, 1), "default": None, "long": (n + 1, n + 2, n + 1)}
    next_type = {0: 1, 1: 4, 4: 5, 5: 7, 7: 0}

    def run(fname, cols, ks, ints, n_out):
        return _call(eng, fname, [_In(_poison(x, k), k) for x, k in zip(cols, ks)], ints, (), n_out)

    def expect(where, rc, got, reff, ints):
        try:
            ref = reff()
        except pqo.OracleError:
            assert rc == ERR_NULLS, f"{where}: the reference fails, the product returned {rc}"
            return
        if _refused_long_window(rc, ints, n, where):
            return
        assert rc == 0, f"{where}: rc {rc}: {_L().pqb_last_error().decode()}"
        _same(where, got, ref)

    for iname, oks in inputs.items():
        K = [oks.get(f) for f in "hlc"]
        for pname, pp in periods.items():
            fk, sk, sd = pp or (5, 3, 3)
            for m1 in MATYPES:
                for m2 in MATYPES:
                    P = (fk, sk, m1, sd, m2)
                    rc, got = run("pqb_stoch_ma", (h, l, c), K, P, 2)
                    expect(f"STOCH{P} n={n} {iname}", rc, got, lambda: pqo.stoch(h, l, c, *P, *K), (fk, sk, sd))
                P = (fk, 3 if pp is None else pp[1], m1)
                rc, got = run("pqb_stochf", (h, l, c), K, P, 2)
                expect(f"STOCHF{P} n={n} {iname}", rc, got, lambda: pqo.stochf(h, l, c, *P, *K), P[:2])
                f_, s_, g_ = pp or (12, 26, 9)
                for ms in ((m1, m1, m1), (m1, next_type[m1], 7), (5, m1, next_type[m1])):
                    P = (f_, ms[0], s_, ms[1], g_, ms[2])
                    rc, got = run("pqb_macdext", (c,), [K[2]], P, 3)
                    expect(f"MACDEXT{P} n={n} {iname}", rc, got, lambda: pqo.macdext(c, *P, ok=K[2]), (f_, s_, g_))
            for m in REFUSED:
                assert run("pqb_stoch_ma", (h, l, c), K, (fk, sk, m, sd, 0), 2)[0] == ERR_UNSUPPORTED
                assert run("pqb_stoch_ma", (h, l, c), K, (fk, sk, 1, sd, m), 2)[0] == ERR_UNSUPPORTED
                assert run("pqb_stochf", (h, l, c), K, (fk, 3, m), 2)[0] == ERR_UNSUPPORTED
                assert run("pqb_macdext", (c,), [None], (12, m, 26, 0, 9, 0), 3)[0] == ERR_UNSUPPORTED
                assert run("pqb_macdext", (c,), [None], (12, 0, 26, 0, 9, m), 3)[0] == ERR_UNSUPPORTED
    # STOCHRSI: clean, flat stretches (RSI 0 / 100 and zero-range %K windows), and nulls (RSI refuses them)
    for cname, x in (("random walk", c), ("flat stretches", _flat_prices(n, seed=n))):
        for tp, fk, fd in ((14, 5, 3), (1, 1, 1), (n + 1, n + 1, n + 1), (3, 4, 2)):
            for m in MATYPES:
                rc, got = run("pqb_stochrsi", (x,), [None], (tp, fk, fd, m), 2)
                expect(f"STOCHRSI({tp},{fk},{fd},{m}) n={n} {cname}", rc, got, lambda: pqo.stochrsi(x, tp, fk, fd, m),
                       (tp, fk, fd))
        for m in REFUSED:
            assert run("pqb_stochrsi", (x,), [None], (14, 5, 3, m), 2)[0] == ERR_UNSUPPORTED
    if n > 1:
        rc, _ = run("pqb_stochrsi", (c,), [holes], (14, 5, 3, 0), 2)
        assert rc == ERR_NULLS
        with pytest.raises(pqo.OracleError):
            pqo.stochrsi(c, 14, 5, 3, 0, ok=holes)


# ---- concurrency -----------------------------------------------------------------------------------------------------------
def test_many_threads_on_one_engine_across_lengths(pq):
    """16 threads on one engine, each looping over its own mix of lengths on both sides of 32,768: MACDEXT (whose col_sub pass
    runs outside the engine's lock), STOCHRSI and null-bearing SMA.  Every result equals the same call made serially."""
    e = pq.Engine(0)
    try:
        jobs = []
        for t in range(16):
            mix = []
            for j, n in enumerate((300 + t, 32_768 - t % 2, 32_769 + t, 1000 + 8 * t + 5)):
                x = _flat_prices(n, seed=100 * t + j) if (t + j) % 3 == 0 else synth.ohlcv(1, n, seed=100 * t + j)["close"][0]
                ok = np.random.default_rng(t * 7 + j).random(n) > 0.05
                mt = MATYPES[(t + j) % len(MATYPES)]
                mix += [("pqb_macdext", [_In(x)], (5 + t % 7, mt, 20, MATYPES[(t + 2 * j) % 5], 4 + j, MATYPES[j % 5]), 3),
                        ("pqb_stochrsi", [_In(x)], (14, 3 + t % 5, 3, MATYPES[t % 5]), 2),
                        ("pqb_sma", [_In(_poison(x, ok), ok)], (3 + t,), 1)]
            jobs.append(mix)
        serial = [[_call(e, f, ins, ints, (), n_out) for f, ins, ints, n_out in mix] for mix in jobs]
        assert all(rc == 0 for s in serial for rc, _ in s)
        errors = []

        def work(t):
            try:
                for _ in range(3):
                    for (f, ins, ints, n_out), (_, ref) in zip(jobs[t], serial[t]):
                        rc, got = _call(e, f, ins, ints, (), n_out)
                        assert rc == 0, f"thread {t} {f}: rc {rc}"
                        for (gv, gk), (rv, rk) in zip(got, ref):
                            assert np.array_equal(gk, rk), f"thread {t} {f} {ints}: validity differs from the serial call"
                            assert T.same_bits(gv, rv).all(), f"thread {t} {f} {ints}: values differ from the serial call"
            except Exception as ex:                       # noqa: BLE001
                errors.append(ex)

        ts = [threading.Thread(target=work, args=(t,)) for t in range(16)]
        [t.start() for t in ts]
        [t.join() for t in ts]
        assert not errors, errors[:3]
    finally:
        e.close()
