"""The optional indicator groups (outputs 21-42) on panels with halts, delistings, late listings and fields that start on
different rows, against the oracle's null rules, bit for bit in values and validity:
- midpoint and adosc skip null bars (overlap.rs / volume.rs);
- the momentum.rs functions (mom, the roc family, cmo, trix, cci, the DM family, ultosc, mfi, aroon) make the whole column
  null for a symbol with a null after a field's first valid bar, in any field they read; the Donchian lines follow
  midprice's rule (high / low);
- with leading nulls only, their series starts at the first bar where every field they read is valid."""
import ctypes as C

import numpy as np
import pytest

import synth
import tolerances as T
from oracle import pqo

pytestmark = pytest.mark.gpu

F = ("close", "high", "low", "volume")
DM_OUT = ("plus_dm", "minus_dm", "dx", "minus_di", "adx", "adxr")
READS = {"mom": "c", "roc": "c", "cmo": "c", "trix": "c", "cci": "hlc", "dm": "hlc", "ultosc": "hlc", "mfi": "hlcv",
         "aroon": "hl", "donchian": "hl"}
DEFAULTS = dict(midpoint_period=14, adosc_fast=3, adosc_slow=10, mom_period=10, roc_period=10, cmo_period=14, mfi_period=14,
                cci_period=14, dm_period=14, trix_period=30, ultosc_period1=7, ultosc_period2=14, ultosc_period3=28,
                aroon_period=14, donchian_period=20)
ONES = {k: 1 for k in DEFAULTS}


def _random_periods(seed):
    rng = np.random.default_rng(seed)
    P = {k: int(rng.integers(1, 40)) for k in DEFAULTS}
    P["mom_period"] = 1
    P["donchian_period"] = 1
    return P


def _outputs_of(g):
    return (("roc", "rocp", "rocr", "rocr100") if g == "roc" else DM_OUT if g == "dm" else ("aroon_up", "aroon_down") if g == "aroon"
            else ("donchian_upper", "donchian_lower") if g == "donchian" else (g,))


def _oracle(g, c, h, l, v, P):
    """{output: (values, validity)} of group g over one symbol's dense series."""
    if g == "mom":
        return {"mom": pqo.mom(c, P["mom_period"])}
    if g == "roc":
        return {name: pqo.roc(c, P["roc_period"], kind) for kind, name in enumerate(("roc", "rocp", "rocr", "rocr100"))}
    if g == "cmo":
        return {"cmo": pqo.cmo(c, P["cmo_period"])}
    if g == "trix":
        return {"trix": pqo.trix(c, P["trix_period"])}
    if g == "cci":
        return {"cci": pqo.cci(h, l, c, P["cci_period"])}
    if g == "dm":
        return dict(pqo.dm(h, l, c, P["dm_period"]))
    if g == "ultosc":
        return {"ultosc": pqo.ultosc(h, l, c, P["ultosc_period1"], P["ultosc_period2"], P["ultosc_period3"])}
    if g == "mfi":
        return {"mfi": pqo.mfi(h, l, c, v, P["mfi_period"])}
    if g == "aroon":
        up, dn = pqo.aroon(h, l, P["aroon_period"])
        return {"aroon_up": up, "aroon_down": dn}
    up, lo = pqo.donchian(h, l, P["donchian_period"])
    return {"donchian_upper": up, "donchian_lower": lo}


def expected(d, ok, s, P):
    """Every optional output of symbol s under the reference's null rules."""
    n = d["close"].shape[1]
    c, h, l, v = (np.ascontiguousarray(d[f][s]) for f in F)
    kc, kh, kl, kv = (np.ascontiguousarray(ok[f][s]).astype(np.uint8) for f in F)
    out = {"midpoint": pqo.midpoint(c, P["midpoint_period"], kc),
           "adosc": pqo.adosc(h, l, c, v, P["adosc_fast"], P["adosc_slow"], kh, kl, kc, kv)}
    first = {f[0]: (int(np.argmax(ok[f][s])) if ok[f][s].any() else None) for f in F}
    flagged = {f[0]: first[f[0]] is not None and not ok[f][s][first[f[0]]:].all() for f in F}
    for g, fields in READS.items():
        a = None if any(first[x] is None for x in fields) else max(first[x] for x in fields)
        if a is None or any(flagged[x] for x in fields):
            for name in _outputs_of(g):
                out[name] = (np.full(n, np.nan), np.zeros(n, bool))
            continue
        for name, (rv, rk) in _oracle(g, c[a:], h[a:], l[a:], v[a:], P).items():
            fv, fk = np.full(n, np.nan), np.zeros(n, bool)
            fv[a:], fk[a:] = rv, rk
            out[name] = (fv, fk)
    return out


def null_patterns(S, N, seed):
    """One null pattern per symbol, cycling: none; shared leading nulls; volume / high starting later; a single interior null
    in close / high / low / volume; clustered halts; an all-field halt; delisted; never listed."""
    rng = np.random.default_rng(seed)
    ok = {f: np.ones((S, N), bool) for f in F}
    for s in range(S):
        kind = s % 12
        t = int(rng.integers(50, N - 50))
        if kind == 1:
            for f in F: ok[f][s, :t] = False
        elif kind == 2:
            ok["volume"][s, :t] = False
        elif kind == 3:
            ok["high"][s, :t] = False
        elif 4 <= kind <= 7:
            ok[F[kind - 4]][s, t] = False
        elif kind == 8:
            for q in range(3):
                u = int(rng.integers(20, N - 10))
                ok["close"][s, u:u + 3] = False
        elif kind == 9:
            for f in F: ok[f][s, t:t + 5] = False
        elif kind == 10:
            for f in F: ok[f][s, t:] = False
        elif kind == 11:
            for f in F: ok[f][s] = False
    return ok


def panel_with_nulls(pq, d, ok, outputs_mask):
    S, N = d["close"].shape
    panel = pq.Panel(S, N, outputs_mask=outputs_mask)
    for s in range(S):
        for f in F:
            bits = None if ok[f][s].all() else np.packbits(ok[f][s].astype(np.uint8), bitorder="little")
            panel.set_column(s, f, d[f][s], validity=bits)
    return panel


def _copy(res):
    return {k: (v.copy(), m.copy()) for k, (v, m) in res.items()}


def _same(a, b, name, rows=slice(None)):
    assert np.array_equal(a[name][1][rows], b[name][1][rows]), name
    assert T.same_bits(a[name][0][rows], b[name][0][rows]).all(), name


EXTRA_NAMES = ("midpoint", "adosc", "mom", "roc", "rocp", "rocr", "rocr100", "cmo", "mfi", "cci") + DM_OUT + (
    "trix", "ultosc", "aroon_up", "aroon_down", "donchian_upper", "donchian_lower")


@pytest.mark.parametrize("periods", ["default", "ones", "random"])
def test_every_optional_group_on_every_null_pattern(periods):
    import polars_quant_b200 as pq
    from polars_quant_b200 import _native as N
    P = dict(DEFAULTS) if periods == "default" else dict(ONES) if periods == "ones" else _random_periods(5)
    S, NB = 40, 700
    d = synth.ohlcv(S, NB, seed=41)
    ok = null_patterns(S, NB, seed=17)
    panel = panel_with_nulls(pq, d, ok, (1 << N.N_OUTPUTS) - 1)
    extras = sum(N.IND_EXTRA.values())
    suite = _copy(panel.compute(N.default_params(indicators=N.IND_ALL, **P)))
    res = _copy(panel.compute(N.default_params(indicators=extras | N.IND_ALL, **P)))
    alone = _copy(panel.compute(N.default_params(indicators=extras, **P)))
    for s in range(S):
        for name, (v, k) in expected(d, ok, s, P).items():
            for got in (res, alone):
                nbad, msg = T.compare(name, got[name][0][s], got[name][1][s], v, k)
                assert nbad == 0, f"symbol {s} (pattern {s % 12}): {msg}"
    for name in pqo.OUTPUT_NAMES:                            # the benchmark outputs do not notice the optional groups
        _same(suite, res, name)
    panel.close()


def test_single_groups_dm_and_cci_on_halted_symbols():
    import polars_quant_b200 as pq
    from polars_quant_b200 import _native as N
    S, NB = 40, 700
    d = synth.ohlcv(S, NB, seed=3)
    ok = null_patterns(S, NB, seed=9)
    panel = panel_with_nulls(pq, d, ok, (1 << N.N_OUTPUTS) - 1)
    for g in ("dm", "cci", "midpoint", "adosc", "mfi"):
        res = panel.compute(N.default_params(indicators=N.IND_EXTRA[g], **DEFAULTS))
        for s in range(S):
            exp = expected(d, ok, s, DEFAULTS)
            for name in _outputs_of(g):
                nbad, msg = T.compare(name, res[name][0][s], res[name][1][s], *exp[name])
                assert nbad == 0, f"group {g} symbol {s}: {msg}"
    panel.close()


def test_multi_wave_panel_with_a_few_halted_symbols():
    """5,120 symbols (several waves), 3 % of them halted: the benchmark outputs are byte-identical to a run of the benchmark groups
    alone, and the unflagged symbols' optional outputs to the same panel without the nulls; run_host equals compute."""
    import polars_quant_b200 as pq
    from polars_quant_b200 import _native as N
    S, NB = 5120, 400
    d = synth.ohlcv(S, NB, seed=23)
    rng = np.random.default_rng(8)
    halted = np.sort(rng.choice(S, S * 3 // 100, replace=False))
    ok = {f: np.ones((S, NB), bool) for f in F}
    for i, s in enumerate(halted):
        t = int(rng.integers(30, NB - 10))
        if i % 3 == 0:
            ok["close"][s, t:t + 3] = False
        elif i % 3 == 1:
            for f in F: ok[f][s, t:t + 3] = False
        else:
            for f in F: ok[f][s, t:] = False
    mask = (1 << N.N_OUTPUTS) - 1
    extras = sum(N.IND_EXTRA.values())
    halted_panel = panel_with_nulls(pq, d, ok, mask)
    suite = _copy(halted_panel.compute(N.default_params(indicators=N.IND_ALL)))
    res = _copy(halted_panel.compute(N.default_params(indicators=extras | N.IND_ALL)))
    for name in pqo.OUTPUT_NAMES:
        _same(suite, res, name)
    halted_panel.run_host(N.default_params(indicators=extras | N.IND_ALL), chunk_symbols=32)
    host = halted_panel.outputs()
    for name in tuple(pqo.OUTPUT_NAMES) + EXTRA_NAMES:
        _same(res, host, name)
    for s in halted[::11]:
        for name, (v, k) in expected(d, ok, s, DEFAULTS).items():
            nbad, msg = T.compare(name, res[name][0][s], res[name][1][s], v, k)
            assert nbad == 0, f"symbol {s}: {msg}"
    halted_panel.close()
    clean_panel = pq.Panel(S, NB, outputs_mask=mask)
    clean_panel.set_fields(d["close"], d["high"], d["low"], d["volume"])
    clean = _copy(clean_panel.compute(N.default_params(indicators=extras | N.IND_ALL)))
    clean_panel.close()
    unflagged = np.setdiff1d(np.arange(S), halted)
    for name in EXTRA_NAMES:
        _same(clean, res, name, unflagged)


def test_wide_table_and_multi_gpu_driver_with_null_cells():
    import pyarrow as pa
    import polars_quant_b200 as pq
    from polars_quant_b200 import _native as N, wide
    S, NB = 40, 500
    d = synth.ohlcv(S, NB, seed=61)
    ok = null_patterns(S, NB, seed=2)
    mask = (1 << N.N_OUTPUTS) - 1
    params = N.default_params(indicators=sum(N.IND_EXTRA.values()) | N.IND_ALL)
    panel = panel_with_nulls(pq, d, ok, mask)
    ref = _copy(panel.compute(params))
    panel.close()
    syms = [f"S{s:03d}" for s in range(S)]
    cols = {"date": pa.array(np.arange(NB, dtype=np.int64))}
    for s, sym in enumerate(syms):
        for f in F:
            cols[f"{sym}_{f}"] = pa.array(d[f][s], type=pa.float64(), mask=~ok[f][s])
    out = wide.WidePanel(pa.table(cols)).suite(params, outputs=list(EXTRA_NAMES) + ["sma", "rsi", "atr"])
    for s, sym in enumerate(syms):
        for name in EXTRA_NAMES + ("sma", "rsi", "atr"):
            a = out[f"{sym}_{name}"].combine_chunks()
            gk = ~np.asarray(a.is_null())
            gv = np.asarray(a.to_numpy(zero_copy_only=False), dtype=np.float64)
            assert np.array_equal(gk, ref[name][1][s]), (sym, name)
            assert T.same_bits(gv[gk], ref[name][0][s][gk]).all(), (sym, name)
    import torch
    if torch.cuda.device_count() < 2:
        return
    mp = pq.MultiPanel(S, NB, list(range(torch.cuda.device_count())), outputs_mask=mask)
    for s in range(S):
        for f in F:
            mp.set_column(s, f, d[f][s], None if ok[f][s].all() else np.packbits(ok[f][s].astype(np.uint8), bitorder="little"))
    mp.run_host(params)
    for s in range(S):
        for k, name in enumerate(N.OUTPUT_NAMES):
            if name in EXTRA_NAMES or name in pqo.OUTPUT_NAMES:
                v, m = mp.get_output(s, k)
                assert np.array_equal(m, ref[name][1][s]), (s, name)
                assert T.same_bits(v[m], ref[name][0][s][m]).all(), (s, name)
    mp.close()


def test_single_column_midpoint_and_adosc_skip_nulls_and_momentum_entry_points_refuse():
    import pyarrow as pa
    import polars_quant_b200 as pq
    from polars_quant_b200 import _native as N, talib
    L = N.lib()
    eng = pq.get_engine(0)
    n = 600
    d = synth.ohlcv(1, n, seed=19)
    c, h, l, v = (np.ascontiguousarray(d[f][0]) for f in F)
    rng = np.random.default_rng(6)
    oks = {f: rng.random(n) > 0.06 for f in F}
    oks["close"][:12] = False
    oks["volume"][n - 30:] = False
    bits = {f: np.packbits(oks[f].astype(np.uint8), bitorder="little") for f in F}
    col = lambda a, f: N.Col(a.ctypes.data, bits[f].ctypes.data, 0, n)
    out_v, out_b = np.empty(n), np.zeros((n + 7) // 8, np.uint8)
    oc = N.OutCol(out_v.ctypes.data, out_b.ctypes.data)
    got = lambda: (out_v.copy(), np.unpackbits(out_b, bitorder="little")[:n].astype(bool))
    cc, ch, cl, cv = col(c, "close"), col(h, "high"), col(l, "low"), col(v, "volume")
    kc, kh, kl, kv = (oks[f].astype(np.uint8) for f in F)
    for p in (1, 2, 14, 90):
        N.check(L.pqb_midpoint(eng._h, C.byref(cc), p, C.byref(oc)))
        assert T.compare("midpoint", *got(), *pqo.midpoint(c, p, kc))[0] == 0
        arr = talib.MIDPOINT(pa.array(c, mask=~oks["close"]), p)
        assert T.compare("midpoint", np.asarray(arr.to_numpy(zero_copy_only=False), dtype=np.float64),
                         ~np.asarray(arr.is_null()), *pqo.midpoint(c, p, kc))[0] == 0
    for fp, sp in ((3, 10), (1, 1), (12, 5)):
        N.check(L.pqb_adosc(eng._h, C.byref(ch), C.byref(cl), C.byref(cc), C.byref(cv), fp, sp, C.byref(oc)))
        ref = pqo.adosc(h, l, c, v, fp, sp, kh, kl, kc, kv)
        assert T.compare("adosc", *got(), *ref)[0] == 0
        arr = talib.ADOSC(*(pa.array(x, mask=~oks[f]) for x, f in ((h, "high"), (l, "low"), (c, "close"), (v, "volume"))), fp, sp)
        assert T.compare("adosc", np.asarray(arr.to_numpy(zero_copy_only=False), dtype=np.float64),
                         ~np.asarray(arr.is_null()), *ref)[0] == 0
    # the momentum.rs entry points still fail on any null, as the reference's cont_slice()? does
    assert L.pqb_mom(eng._h, C.byref(cc), 10, C.byref(oc)) == -5
    assert L.pqb_roc(eng._h, C.byref(cc), 10, 0, C.byref(oc)) == -5
    assert L.pqb_cmo(eng._h, C.byref(cc), 14, C.byref(oc)) == -5
    assert L.pqb_mfi(eng._h, C.byref(ch), C.byref(cl), C.byref(cc), C.byref(cv), 14, C.byref(oc)) == -5
    assert L.pqb_cci(eng._h, C.byref(ch), C.byref(cl), C.byref(cc), 14, C.byref(oc)) == -5


@pytest.mark.parametrize("tag", ["B", "Bs"])
def test_executed_reference_midpoint_and_adosc_with_interior_nulls(tag):
    """The executed-reference vectors of midpoint and adosc on inputs with interior nulls (tags B and Bs), bit for bit
    (midpoint: bars whose window holds a NaN value left out, as in test_gpu_ref_golden)."""
    pytest.importorskip("pyarrow")
    import refgolden
    from test_gpu_ref_golden import _np, _windows_without_nan, gpu_call
    g, index = refgolden.load()
    n_checked = 0
    for e in index:
        if e["tag"] != tag or e["fn"] not in ("midpoint", "adosc"):
            continue
        cols = refgolden.inputs(g, e)
        want = refgolden.expected(g, e)
        assert want is not None, e["key"]
        got = gpu_call(e, cols)
        for arr, (gv, gok) in zip(got, want):
            vals, ok = _np(arr)
            if e["fn"] == "midpoint":
                keep = _windows_without_nan(cols, e)
                vals, ok, gv, gok = vals[keep], ok[keep], gv[keep], gok[keep]
            msg = refgolden.same(vals, ok, gv, gok)
            assert not msg, f"{tag}/{e['key']}: {msg}"
        n_checked += 1
    assert n_checked >= 7, n_checked                       # five midpoint periods and two adosc calls
