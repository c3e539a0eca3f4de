#!/usr/bin/env python
"""Golden vectors for SURVEY.md 8(a): outputs of the REFERENCE ITSELF, made by executing its own source text.

The reference (Rust crate + polars plugin) cannot be built or imported in this image (no cargo / rustc /
maturin / polars; the snapshot does not even type-check -- SURVEY.md facts 2-3).  Its indicator functions are,
however, plain scalar loops in a small subset of Rust, so this script runs them with the interpreter in
tests/golden/rustexec/ (parser + evaluator + a model of the few polars / std containers they touch):

    src/talib/{overlap,momentum,volatility,volume,price}.rs      -- read at generation time
    python/polars_quant/talib/*.py                               -- imported verbatim

Every vector below is therefore the reference's own arithmetic in the reference's own operation order (IEEE
f64, true fma for mul_add, release-profile usize wrap-around), including its panics (`err` = 2: the process
would abort) and its PolarsResult errors (`err` = 1).  The only definitions that are NOT reference text are
the frozen decisions D1 (calc_rma, undefined in the snapshot) and D2 (slice-style calc_ema / calc_sma), see
rustexec/ref_exec.py; the functions that go through D1 are listed in `d1_functions` inside the file.

Run with POLARS_QUANT_REFERENCE set to a checkout of the original polars-quant (the paths above are relative to it):
    python tests/golden/make_ref_golden.py            # writes tests/golden/talib_ref_golden.npz
    python tests/golden/make_ref_golden.py --check    # re-executes and compares with the committed file
"""
from __future__ import annotations

import json
import sys
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
ROOT = HERE.parents[1]
sys.path.insert(0, str(HERE))
sys.path.insert(0, str(ROOT / "tests"))

from rustexec.py_shims import Expr, Shims  # noqa: E402
from rustexec.ref_exec import Reference, ReferenceError, ReferencePanic, column, series  # noqa: E402
import synth  # noqa: E402

OUT = HERE / "talib_ref_golden.npz"

D1_FUNCTIONS = ["adx", "adxr", "dx", "minus_di", "minus_dm", "plus_di", "plus_dm", "rsi", "STOCHRSI"]


# ---------------------------------------------------------------------------------------------------
# input cases
# ---------------------------------------------------------------------------------------------------
def cases():
    """-> {tag: dict(cols={name: (values, validity|None)}, chunks=[...]|None, force_bitmap=bool)}"""
    out = {}
    d = synth.ohlcv(1, 252, seed=0xC0FFEE)
    out["A"] = dict(cols={k: (d[k][0], None) for k in d})                         # config 1: 1 x 252, dense

    d = synth.ohlcv(1, 300, seed=11)
    rng = np.random.Generator(np.random.Philox(12))
    cols = {}
    for k in d:
        ok = rng.random(300) > 0.03
        ok[:3] = False                                                             # a later listing
        cols[k] = (d[k][0], ok)
    out["B"] = dict(cols=cols)                                                     # nulls, different per field

    d = synth.ohlcv(1, 300, seed=13)
    ok = np.ones(300, bool)
    ok[:7] = False
    ok[120:123] = False
    ok[290:] = False
    out["Bs"] = dict(cols={k: (d[k][0], ok.copy()) for k in d})                   # nulls shared by all fields

    d = synth.ohlcv(1, 252, seed=0xC0FFEE)
    out["C3"] = dict(cols={k: (d[k][0], None) for k in d}, chunks=[100, 1, 151])   # 3 chunks: state carries over
    out["Cb"] = dict(cols={k: (d[k][0], None) for k in d}, force_bitmap=True)      # dense, bitmap present

    # coarse grid: flat windows (0/0), closes on the extremes, zero volume, repeated values
    rng = np.random.Generator(np.random.Philox(21))
    n = 280
    c = 50.0 + np.cumsum(rng.integers(-2, 3, n)) * 0.5
    c[40:75] = c[40]
    o = np.concatenate([[c[0]], c[:-1]])
    h = np.maximum(o, c) + rng.integers(0, 2, n) * 0.5
    lo = np.minimum(o, c) - rng.integers(0, 2, n) * 0.5
    h[40:75] = c[40]
    lo[40:75] = c[40]
    v = np.round(rng.lognormal(8.0, 1.0, n))
    v[rng.random(n) < 0.1] = 0.0
    out["D"] = dict(cols=dict(open=(o, None), high=(h, None), low=(lo, None), close=(c, None), volume=(v, None)))

    for n in (0, 1, 2, 10):                                                        # the guards
        d = synth.ohlcv(1, max(n, 1), seed=30 + n)
        out[f"E{n}"] = dict(cols={k: (d[k][0][:n], None) for k in d})

    # NaN / inf VALUES (not nulls): the reference treats them as numbers (SURVEY.md 8a)
    d = synth.ohlcv(1, 200, seed=41)
    cols = {k: d[k][0].copy() for k in d}
    cols["close"][50] = np.nan
    cols["high"][90] = np.nan
    cols["low"][130] = np.nan
    cols["high"][131] = np.nan
    cols["volume"][20] = np.nan
    cols["close"][170] = np.inf
    out["F"] = dict(cols={k: (x, None) for k, x in cols.items()})

    d = synth.ohlcv(1, 700, seed=51)
    out["G"] = dict(cols={k: (d[k][0], None) for k in d})                         # long windows (config 5)
    return out


# ---------------------------------------------------------------------------------------------------
# the calls
# ---------------------------------------------------------------------------------------------------
def call_table(tag):
    """-> list of (key, kind, fn, column names, params/kwargs).  kind 'rs' = a Rust plugin fn, 'py' = a Python
    shim composition."""
    t = []
    rs = lambda key, fn, cols, params=(), **kw: t.append(dict(key=key, kind="rs", fn=fn, cols=cols, params=list(params), kwargs=kw))
    py = lambda key, mod, fn, cols, *params: t.append(dict(key=key, kind="py", mod=mod, fn=fn, cols=cols, params=list(params)))
    periods = (1, 2, 5, 30) if tag != "G" else (55, 250)
    for p in periods:
        for fn in ("sma", "ema", "tema", "trima", "wma", "dema", "kama"):
            rs(f"{fn}_{p}", fn, ["close"], timeperiod=p)
        rs(f"t3_{p}", "t3", ["close"], timeperiod=p, vfactor=0.7)
        rs(f"midpoint_{p}", "midpoint", ["close"], timeperiod=p)
        rs(f"midprice_{p}", "midprice", ["high", "low"], timeperiod=p)
        rs(f"willr_{p}", "willr", ["high", "low", "close"], [p])
        rs(f"atr_{p}", "atr", ["high", "low", "close"], timeperiod=p)
        rs(f"rsi_{p}", "rsi", ["close"], [p])
        rs(f"aroon_{p}", "aroon", ["high", "low"], [p])
        py(f"STOCH_{p}_3_3", "momentum", "STOCH", ["high", "low", "close"], p, 3, 0, 3, 0)
    rs("t3_5_v0", "t3", ["close"], timeperiod=5, vfactor=0.0)
    rs("trima_7", "trima", ["close"], timeperiod=7)
    rs("trima_8", "trima", ["close"], timeperiod=8)
    for mt in range(9):
        rs(f"ma_5_{mt}", "ma", ["close"], timeperiod=5, matype=mt)
    rs("sma_default", "sma", ["close"])
    rs("bbands_default", "bbands", ["close"])
    rs("bbands_20", "bbands", ["close"], timeperiod=20, nbdevup=2.0, nbdevdn=2.0)
    rs("bbands_5", "bbands", ["close"], timeperiod=5, nbdevup=1.5, nbdevdn=2.5)
    rs("macd_12_26_9", "macd", ["close"], [12, 26, 9])
    rs("macd_3_5_8", "macd", ["close"], [3, 5, 8])
    rs("macd_5_3_2", "macd", ["close"], [5, 3, 2])
    rs("trange", "trange", ["high", "low", "close"])
    rs("natr_14", "natr", ["high", "low", "close"], timeperiod=14)
    rs("atr_default", "atr", ["high", "low", "close"])
    rs("obv", "obv", ["close", "volume"])
    rs("ad", "ad", ["high", "low", "close", "volume"])
    rs("adosc_3_10", "adosc", ["high", "low", "close", "volume"], fastperiod=3, slowperiod=10)
    rs("adosc_default", "adosc", ["high", "low", "close", "volume"])
    rs("willr_14", "willr", ["high", "low", "close"], [14])
    rs("midprice_14", "midprice", ["high", "low"], timeperiod=14)
    rs("midpoint_14", "midpoint", ["close"], timeperiod=14)
    rs("rsi_14", "rsi", ["close"], [14])
    rs("mom_10", "mom", ["close"], [10])
    for fn in ("roc", "rocp", "rocr", "rocr100"):
        rs(f"{fn}_10", fn, ["close"], [10])
    rs("cmo_14", "cmo", ["close"], [14])
    rs("mfi_14", "mfi", ["high", "low", "close", "volume"], [14])
    rs("cci_14", "cci", ["high", "low", "close"], [14])
    rs("cci_5", "cci", ["high", "low", "close"], [5])
    for fn in ("adx", "adxr", "dx", "minus_di", "plus_di"):
        rs(f"{fn}_14", fn, ["high", "low", "close"], [14])
    for fn in ("minus_dm", "plus_dm"):
        rs(f"{fn}_14", fn, ["high", "low"], [14])
    rs("trix_30", "trix", ["close"], [30])
    rs("trix_5", "trix", ["close"], [5])
    rs("ultosc_7_14_28", "ultosc", ["high", "low", "close"], [7, 14, 28])
    rs("ultosc_3_5_9", "ultosc", ["high", "low", "close"], [3, 5, 9])
    rs("aroon_14", "aroon", ["high", "low"], [14])
    rs("bop", "bop", ["open", "high", "low", "close"])
    rs("avgprice", "avgprice", ["open", "high", "low", "close"])
    rs("medprice", "medprice", ["high", "low"])
    rs("typprice", "typprice", ["high", "low", "close"])
    rs("wclprice", "wclprice", ["high", "low", "close"])
    py("STOCH_5_3_3", "momentum", "STOCH", ["high", "low", "close"], 5, 3, 0, 3, 0)
    py("STOCH_9_3_3", "momentum", "STOCH", ["high", "low", "close"], 9, 3, 0, 3, 0)       # KDJ's K and D (D3)
    py("STOCH_14_5_1_4_1", "momentum", "STOCH", ["high", "low", "close"], 14, 5, 1, 4, 1)  # EMA smoothing
    py("STOCHF_5_3", "momentum", "STOCHF", ["high", "low", "close"], 5, 3, 0)
    py("STOCHRSI_14_5_3", "momentum", "STOCHRSI", ["close"], 14, 5, 3, 0)
    py("MACDEXT_12_0_26_0_9_0", "momentum", "MACDEXT", ["close"], 12, 0, 26, 0, 9, 0)
    py("MACDEXT_12_1_26_1_9_1", "momentum", "MACDEXT", ["close"], 12, 1, 26, 1, 9, 1)
    py("MACDFIX_9", "momentum", "MACDFIX", ["close"], 9)
    return t


def has_nan(case, names):
    return any(np.isnan(case["cols"][k][0]).any() or np.isinf(case["cols"][k][0]).any() for k in names)


def generate():
    ref = Reference()
    shims = Shims(ref)
    arrays, index = {}, []
    for tag, case in cases().items():
        for k, (x, ok) in case["cols"].items():
            arrays[f"{tag}/in/{k}"] = np.asarray(x, dtype=np.float64)
            if ok is not None:
                arrays[f"{tag}/in/{k}_ok"] = ok
        meta = dict(chunks=case.get("chunks"), force_bitmap=bool(case.get("force_bitmap", False)))
        mk = lambda name: series(case["cols"][name][0], case["cols"][name][1], case.get("chunks"),
                                 force_bitmap=case.get("force_bitmap", False))
        for call in call_table(tag):
            key = f"{tag}/{call['key']}"
            entry = dict(call, tag=tag, **meta)
            if call["kind"] == "py" and has_nan(case, call["cols"]):
                continue                                    # polars' NaN ordering in rolling windows: not modelled
            try:
                if call["kind"] == "rs":
                    res = ref.call(call["fn"], [mk(c) for c in call["cols"]], call["params"], call["kwargs"])
                else:
                    f = getattr(getattr(shims.talib, call["mod"]), call["fn"])
                    r = f(*[Expr(mk(c).inner) for c in call["cols"]], *call["params"])
                    res = [column(e.ca) for e in (r if isinstance(r, tuple) else (r,))]
                for j, (vals, ok) in enumerate(res):
                    arrays[f"{key}/{j}/v"] = vals
                    arrays[f"{key}/{j}/ok"] = ok
                entry["n_out"] = len(res)
            except ReferenceError:
                arrays[f"{key}/err"] = np.array([1])
                entry["err"] = 1
            except ReferencePanic:
                arrays[f"{key}/err"] = np.array([2])
                entry["err"] = 2
            index.append(entry)
    arrays["index"] = np.array(json.dumps(index))
    arrays["d1_functions"] = np.array(D1_FUNCTIONS)
    return arrays


def main():
    arrays = generate()
    if "--check" in sys.argv:
        old = np.load(OUT)
        bad = [k for k in arrays if k not in old.files or not np.array_equal(
            np.asarray(arrays[k]).view(np.uint8) if np.asarray(arrays[k]).dtype.kind == "f" else arrays[k],
            old[k].view(np.uint8) if old[k].dtype.kind == "f" else old[k])]
        bad += [k for k in old.files if k not in arrays]
        print("differences:", bad[:10], len(bad))
        return 1 if bad else 0
    np.savez_compressed(OUT, **arrays)
    idx = json.loads(str(arrays["index"]))
    print("wrote", OUT, OUT.stat().st_size, "bytes;", len(idx), "calls;",
          sum(1 for e in idx if e.get("err") == 1), "Err;", sum(1 for e in idx if e.get("err") == 2), "panics")
    return 0


if __name__ == "__main__":
    sys.exit(main())
