"""Time-split panels (include/pqb200.h "time-split panels", DESIGN.md section 4c) for every group the whitelist admits, at
ragged shapes, through the C ABI and the benchmarked device path, and with halts at chunk starts.

Two references:
- serial: the oracle on the full row.  Validity exact, values within rel 1e-10 / abs 1e-12; pure window functions and
  chunk 0 bit for bit.
- geometry: DESIGN 4c restated.  Virtual symbol c*S + s holds bars [max(0, c*L - W), ... + vbars) of symbol s, padded
  with its last value; L and W are rounded up to 32 and vbars = min(L + W, round32(n_bars)).  The oracle on those
  virtual rows, spliced by chunk, must equal the split output bit for bit, values and validity.  A symbol whose
  warm-up is too flat for RSI or the DM family in some chunk (fewer moving bars than the warm-up count of its
  periods) is recomputed serially instead: its outputs equal the serial oracle bit for bit."""
import ctypes as C

import numpy as np
import pytest

import devread
import synth
import tolerances as T
from oracle import pqo
from polars_quant_b200 import _native as N

pytestmark = pytest.mark.gpu
REL, ABS = 1e-10, 1e-12
IND = {**N.IND, **N.IND_EXTRA}
DM_OUT = ("plus_dm", "minus_dm", "dx", "minus_di", "adx", "adxr")
OUTPUTS = {"ema": ("ema",), "tema": ("tema",), "macd": ("macd", "macd_signal", "macd_hist"), "rsi": ("rsi",),
           "trange": ("trange",), "atr": ("atr",), "natr": ("natr",), "willr": ("willr",), "midprice": ("midprice",),
           "donchian": ("donchian_upper", "donchian_lower"), "mom": ("mom",), "roc": ("roc", "rocp", "rocr", "rocr100"),
           "trix": ("trix",), "aroon": ("aroon_up", "aroon_down"), "dm": DM_OUT}
SPLITTABLE = tuple(OUTPUTS)
PURE = {"trange", "willr", "midprice", "donchian_upper", "donchian_lower", "mom", "roc", "rocp", "rocr", "rocr100",
        "aroon_up", "aroon_down"}
SHORT = dict(ema_period=4, tema_period=3, macd_fast=3, macd_slow=6, macd_signal=2, rsi_period=2, atr_period=2,
             natr_period=2, willr_period=5, midprice_period=4, donchian_period=3, mom_period=2, roc_period=3,
             trix_period=2, aroon_period=3, dm_period=2)


@pytest.fixture(scope="module")
def pq():
    import polars_quant_b200 as pq
    return pq


def r32(x):
    return (x + 31) // 32 * 32


def geometry(n_bars, chunks, warmup):
    L = r32(-(-n_bars // chunks))
    W = 0 if chunks == 1 else r32(warmup)
    return L, W, min(L + W, r32(n_bars))


def params(groups, **kw):
    return N.default_params(indicators=sum(IND[g] for g in groups), **kw)


def outputs_mask(groups):
    return sum(1 << N.OUTPUT_NAMES.index(o) for g in groups for o in OUTPUTS[g])


def oracle(groups, prm, c, h, l, v):
    """{output: (values, validity)} of the requested groups over one dense row."""
    out = {}
    for g in groups:
        if g == "ema": out["ema"] = pqo.ema(c, prm.ema_period)
        elif g == "tema": out["tema"] = pqo.tema(c, prm.tema_period)
        elif g == "macd": out.update(zip(OUTPUTS["macd"], pqo.macd(c, prm.macd_fast, prm.macd_slow, prm.macd_signal)))
        elif g == "rsi": out["rsi"] = pqo.rsi(c, prm.rsi_period)
        elif g == "trange": out["trange"] = pqo.trange(h, l, c)
        elif g == "atr": out["atr"] = pqo.atr(h, l, c, prm.atr_period)
        elif g == "natr": out["natr"] = pqo.natr(h, l, c, prm.natr_period)
        elif g == "willr": out["willr"] = pqo.willr(h, l, c, prm.willr_period)
        elif g == "midprice": out["midprice"] = pqo.midprice(h, l, prm.midprice_period)
        elif g == "donchian": out.update(zip(OUTPUTS["donchian"], pqo.donchian(h, l, prm.donchian_period)))
        elif g == "mom": out["mom"] = pqo.mom(c, prm.mom_period)
        elif g == "roc": out.update((name, pqo.roc(c, prm.roc_period, k)) for k, name in enumerate(OUTPUTS["roc"]))
        elif g == "trix": out["trix"] = pqo.trix(c, prm.trix_period)
        elif g == "aroon": out.update(zip(OUTPUTS["aroon"], pqo.aroon(h, l, prm.aroon_period)))
        elif g == "dm": out.update(pqo.dm(h, l, c, prm.dm_period))
    return out


def moving_bars(c, h, l):
    """Per bar t >= 1 of a row: (close moved, calc_dm's +DM or -DM is non-zero) against bar t - 1.  A bar with a range but
    no directional move does not count for DM: smoothed TR cancels out of DX."""
    up, dn = h[1:] - h[:-1], l[:-1] - l[1:]
    return c[1:] != c[:-1], ((up > dn) & (up > 0)) | ((dn > up) & (dn > 0))


def too_flat(groups, prm, c, h, l, n_bars, chunks, warmup):
    """True if some chunk c >= 1 with a base past bar 0 has fewer moving bars in its warm-up [base, c*L) -- its first bar,
    the seed, counted as one -- than RSI (29p + 2 changed closes) or the DM family ((29p + 2) + (p + 2) directional moves:
    DX's own, then ADXR's lag) forget their seed in."""
    L, W, _ = geometry(n_bars, chunks, warmup)
    mc, md = moving_bars(c, h, l)
    for k in range(1, chunks):
        base = k * L - W
        if base <= 0 or k * L >= n_bars:
            continue
        if "rsi" in groups and 1 + mc[base:k * L - 1].sum() < 29 * prm.rsi_period + 2:
            return True
        if "dm" in groups and 1 + md[base:k * L - 1].sum() < 30 * prm.dm_period + 4:
            return True
    return False


def split_model(groups, prm, c, h, l, v, chunks, warmup):
    """The oracle on every chunk's virtual row, spliced into the real row (DESIGN 4c)."""
    n = len(c)
    L, W, vbars = geometry(n, chunks, warmup)
    res = {}
    for k in range(chunks):
        t0 = k * L
        if t0 >= n:
            break
        base = max(0, t0 - W)
        rows = []
        for x in (c, h, l, v):
            r = x[base:base + vbars]
            rows.append(np.concatenate([r, np.full(vbars - len(r), r[-1])]))
        m = min(L, n - t0)
        for name, (rv, rk) in oracle(groups, prm, *rows).items():
            fv, fk = res.setdefault(name, (np.full(n, np.nan), np.zeros(n, bool)))
            fv[t0:t0 + m], fk[t0:t0 + m] = rv[t0 - base:t0 - base + m], rk[t0 - base:t0 - base + m]
    return res


def serial_errors(name, got, ref, chunk_bars):
    """Messages for every way the split output misses the serial bar (empty: it meets it)."""
    (gv, gk), (rv, rk) = got, ref
    errs = []
    if not np.array_equal(gk, rk):
        bad = np.flatnonzero(gk != rk)
        errs.append(f"{name}: validity differs at {bad.size} bars (first {bad[:3].tolist()}, split valid {gk[bad[0]]})")
        return errs
    d = np.abs(gv[rk] - rv[rk])
    lim = ABS + REL * np.abs(rv[rk])
    if not (d <= lim).all():
        i = np.flatnonzero(rk)[np.argmax(d - lim)]
        errs.append(f"{name}: {(d > lim).sum()} bars off, worst at bar {i}: {gv[i]!r} vs {rv[i]!r}")
    exact = T.same_bits(gv[rk], rv[rk])
    if name in PURE and not exact.all():
        errs.append(f"{name}: a pure window function differs in its bits at {(~exact).sum()} bars")
    c0 = rk[:chunk_bars]
    if not T.same_bits(gv[:chunk_bars][c0], rv[:chunk_bars][c0]).all():
        errs.append(f"{name}: chunk 0 is not the serial computation bit for bit")
    return errs


def same(got, ref):
    (gv, gk), (rv, rk) = got, ref
    return np.array_equal(gk, rk) and T.same_bits(gv[rk], rv[rk]).all()


def check_split(p, groups, prm, d, chunks, warmup, expect_flat=False, symbols=None):
    """Every output of every symbol of split panel p against the serial bar and the geometry model."""
    S, n = d["close"].shape
    L, W, vbars = geometry(n, chunks, warmup)
    assert (p.chunk_bars, p.warmup, p.virtual_bars, p.virtual_symbols) == (L, W, vbars, S * chunks)
    errs = []
    for s in range(S) if symbols is None else symbols:
        c, h, l, v = (np.ascontiguousarray(d[f][s]) for f in ("close", "high", "low", "volume"))
        flat = too_flat(groups, prm, c, h, l, n, chunks, warmup)
        if not expect_flat:
            assert not flat, f"symbol {s}: the test data was meant to move in every warm-up"
        serial = oracle(groups, prm, c, h, l, v)
        model = serial if flat else split_model(groups, prm, c, h, l, v, chunks, warmup)
        for name in serial:
            got = p.get_output(s, N.OUTPUT_NAMES.index(name))
            errs += [f"symbol {s}: {e}" for e in serial_errors(name, got, serial[name], L)]
            if not same(got, model[name]):
                errs.append(f"symbol {s}: {name} is not the {'serial' if flat else 'virtual-row'} oracle bit for bit")
    assert not errs, "\n".join(errs[:40])


def ohlcv(S, n, seed, levels=(100.0,)):
    d = synth.ohlcv(S, n, seed=seed)
    for s in range(S):
        for f in ("open", "high", "low", "close"):
            d[f][s] *= levels[s % len(levels)] / 100.0
    return d


# ---- 1. every whitelisted group, alone and with EMA / MACD / RSI, at price levels 1e-3, ~100 and 1e5 ---------------------
GROUP_CASES = [("dm", dict(dm_period=p)) for p in (1, 2, 14, 40)] + \
              [("trix", dict(trix_period=p)) for p in (1, 5, 30)] + \
              [("aroon", dict(aroon_period=p)) for p in (1, 14, 40)] + \
              [("donchian", {}), ("donchian", dict(donchian_period=2)), ("mom", {}), ("mom", dict(mom_period=1)),
               ("roc", {}), ("roc", dict(roc_period=1))]


@pytest.mark.parametrize("with_companions", [False, True], ids=["alone", "with_ema_macd_rsi"])
@pytest.mark.parametrize("group,periods", GROUP_CASES, ids=[f"{g}-{'-'.join(map(str, kw.values())) or 'default'}"
                                                            for g, kw in GROUP_CASES])
def test_every_whitelisted_group(pq, group, periods, with_companions):
    S, NB, chunks = 6, 20_003, 8
    groups = (group, "ema", "macd", "rsi") if with_companions else (group,)
    prm = params(groups, **periods)
    d = ohlcv(S, NB, seed=11, levels=(1e-3, 100.0, 1e5))
    if group in ("mom", "roc"):                  # zero closes: the ROC family's own nulls, inside later chunks
        rng = np.random.default_rng(4)
        for s in range(S):
            d["close"][s, rng.integers(3000, NB, 12)] = 0.0
            d["close"][s, NB - 700:NB - 697] = 0.0
    W = pq.SplitPanel.required_warmup(prm)
    assert W > 0
    p = pq.SplitPanel(S, NB, chunks=chunks, warmup=W, outputs_mask=outputs_mask(groups))
    p.set_fields(d["close"], d["high"], d["low"], d["volume"])
    p.run_host(prm)
    check_split(p, groups, prm, d, chunks, W)
    p.close()


def test_whitelist_is_the_documented_fifteen_groups(pq):
    for g in SPLITTABLE:
        assert pq.SplitPanel.required_warmup(params((g,))) > 0, g
    assert pq.SplitPanel.required_warmup(params(SPLITTABLE)) > 0
    for g in set(IND) - set(SPLITTABLE):
        assert pq.SplitPanel.required_warmup(params((g,))) == -1, g


# ---- 2. ragged geometry ----------------------------------------------------------------------------------------------
RAGGED = [  # symbols, bars, chunks, warm-up asked for (None: what the periods need)
    (1, 1, 1, 0),                 # one bar; chunks = 1 forces W = 0
    (5, 31, 1, 500),
    (33, 33, 2, None),            # W > L: chunk 1's base clips to 0
    (5, 1_001, 7, None),          # n_bars not a multiple of 8, 32 or chunks
    (5, 1_001, 16, None),         # L = 64, W = 256: several bases clip to 0
    (1, 1_001, 2, None),          # L + W > round32(n_bars): vbars clipped to the padded row
    (33, 100, 50, None),          # L = 32: chunks 4..49 start past the end of the row
    (5, 20_003, 8, None),
    (1, 20_003, 9, 2_000),
    (33, 4_099, 5, None),         # virtual symbols of different chunks share a 32-symbol block
]


@pytest.mark.parametrize("S,NB,chunks,warmup", RAGGED, ids=[f"{a}x{b}-c{c}-w{w}" for a, b, c, w in RAGGED])
def test_ragged_geometry(pq, S, NB, chunks, warmup):
    prm = params(SPLITTABLE, **SHORT)
    need = pq.SplitPanel.required_warmup(prm)
    W = need if warmup is None else max(warmup, need)
    d = ohlcv(S, NB, seed=NB + chunks, levels=(100.0, 1e-3, 1e5))
    p = pq.SplitPanel(S, NB, chunks=chunks, warmup=W, outputs_mask=outputs_mask(SPLITTABLE))
    p.set_fields(d["close"], d["high"], d["low"], d["volume"])
    p.run_host(prm)
    check_split(p, SPLITTABLE, prm, d, chunks, W)
    p.close()


# ---- 3. C-ABI intake ---------------------------------------------------------------------------------------------------
def test_c_abi_intake(pq):
    lib = N.lib()
    S, NB, chunks = 3, 1_003, 4
    groups = ("ema", "willr", "roc")
    prm = params(groups)
    W = pq.SplitPanel.required_warmup(prm)
    d = ohlcv(S, NB, seed=21)
    ref = pq.SplitPanel(S, NB, chunks=chunks, warmup=W, outputs_mask=outputs_mask(groups))
    ref.set_fields(d["close"], d["high"], d["low"], d["volume"])
    ref.run_host(prm)
    p = pq.SplitPanel(S, NB, chunks=chunks, warmup=W, outputs_mask=outputs_mask(groups))
    off = 13                                               # an Arrow slice: values and bitmap start 13 slots in
    bits = np.full((off + NB + 7) // 8 + 1, 0xFF, np.uint8)
    for s in range(S):
        for f, name in enumerate(("close", "high", "low", "volume")):
            vals = np.concatenate([np.full(off, -7.0), d[name][s]])
            N.check(lib.pqb_split_set_column(p._h, s, f, vals.ctypes.data_as(C.c_void_p), bits.ctypes.data_as(C.c_void_p),
                                             off, NB))
    p.run_host(prm)
    for s in range(S):
        for name in (o for g in groups for o in OUTPUTS[g]):
            k = N.OUTPUT_NAMES.index(name)
            assert same(p.get_output(s, k), ref.get_output(s, k)), name
    vals = np.concatenate([np.full(off, -7.0), d["close"][0]])
    holed = bits.copy()
    t = off + 700
    holed[t // 8] &= ~np.uint8(1 << (t % 8))
    assert lib.pqb_split_set_column(p._h, 0, 0, vals.ctypes.data_as(C.c_void_p), holed.ctypes.data_as(C.c_void_p),
                                    off, NB) == -5              # PQB_ERR_NULLS
    assert b"null-free" in lib.pqb_last_error()
    h = C.c_void_p()
    assert lib.pqb_split_create(pq.get_engine(0)._h, 2, 10, 11, 0, 0xF, 1 << N.OUTPUT_NAMES.index("ema"), 1,
                                C.byref(h)) == -3                # chunks > n_bars: PQB_ERR_INVALID
    assert not h.value
    p.close()
    ref.close()


# ---- 4. the benchmarked device path: pqb_split_fill_synthetic + pqb_split_run ------------------------------------------
DEVICE_SETS = [  # (groups, periods, fields_mask, sigma): scripts/bench_configs.py c3 split, scripts/bench_next_rows.py c5split
    (("ema", "macd"), dict(ema_period=12), 0b0001, 0.0005),
    (("ema", "macd"), dict(ema_period=200), 0b0001, 0.0005),
    (("willr", "midprice"), dict(willr_period=20, midprice_period=20), 0b0111, 0.02),
    (("willr", "midprice"), dict(willr_period=55, midprice_period=55), 0b0111, 0.02),
]


def _inner(pq, sp, outputs_mask):
    h = N.lib().pqb_split_panel(sp._h)
    return pq.Panel._borrowed(h, sp.engine, sp.virtual_symbols, sp.virtual_bars, outputs_mask, True, owner=sp)


@pytest.mark.parametrize("chunks", [16, 64])
@pytest.mark.parametrize("k", range(len(DEVICE_SETS)),
                         ids=["ema12-macd", "ema200-macd", "willr20-midprice20", "willr55-midprice55"])
def test_device_path_of_the_benchmarks(pq, k, chunks):
    groups, periods, fmask, sigma = DEVICE_SETS[k]
    S, NB, seed = 64, 200_000, 3 + k
    lib = N.lib()
    prm = params(groups, **periods)
    om = outputs_mask(groups)
    W = pq.SplitPanel.required_warmup(prm)
    sp = pq.SplitPanel(S, NB, chunks=chunks, warmup=W, fields_mask=fmask, outputs_mask=om)
    sp.fill_synthetic(seed=seed, sigma=sigma)
    N.check(lib.pqb_split_run(sp._h, C.byref(prm)))
    serial = pq.Panel(S, NB, fields_mask=fmask, outputs_mask=om)
    serial.fill_synthetic(seed=seed, sigma=sigma, to_host=True)
    serial.run(prm)
    serial.download()
    serial.sync()
    # inputs: every chunk's virtual rows are the serial panel's bars [base, base + vbars) of the same seed
    inner = _inner(pq, sp, om)
    nb, bp = inner.tiled_shape()
    L, Wv, vbars = sp.chunk_bars, sp.warmup, sp.virtual_bars
    for f in range(4):
        if not fmask >> f & 1:
            continue
        ref = serial.host_field(f)[:, :NB]
        dev = lib.pqb_panel_device_field(inner._h, f)
        rows = np.concatenate([devread.read_block(dev, b, bp, vbars) for b in range(nb)])[:S * chunks]
        for c in range(chunks):
            base = max(0, c * L - Wv)
            m = min(vbars, NB - base)
            if m > 0:
                assert T.same_bits(rows[c * S:(c + 1) * S, :m], ref[:, base:base + m]).all(), (f, c)
    # outputs: downloaded from the virtual panel, against the serial panel's own (bit-exact to the oracle) results
    inner.download()
    inner.sync()
    errs = []
    for name in (o for g in groups for o in OUTPUTS[g]):
        kk = N.OUTPUT_NAMES.index(name)
        rv, rk = serial.host_output(kk), serial.host_validity(kk)
        for s in range(S):
            errs += serial_errors(f"{name}[{s}]", sp.get_output(s, kk), (rv[s], rk[s]), L)
    assert not errs, "\n".join(errs[:20])
    serial.close()
    sp.close()


def _upload_and_run(pq, p, prm):
    """set_column (done) + pqb_panel_upload + pqb_split_run + pqb_panel_download of the virtual panel."""
    lib = N.lib()
    inner = lib.pqb_split_panel(p._h)
    N.check(lib.pqb_panel_upload(inner))
    N.check(lib.pqb_split_run(p._h, C.byref(prm)))
    N.check(lib.pqb_panel_download(inner))
    N.check(lib.pqb_panel_sync(inner))


def test_upload_path_equals_run_host(pq):
    S, NB, chunks = 8, 100_000, 16
    groups = ("ema", "macd", "rsi", "dm", "willr", "roc")
    prm = params(groups)
    W = pq.SplitPanel.required_warmup(prm)
    d = ohlcv(S, NB, seed=31)
    a = pq.SplitPanel(S, NB, chunks=chunks, warmup=W, outputs_mask=outputs_mask(groups))
    b = pq.SplitPanel(S, NB, chunks=chunks, warmup=W, outputs_mask=outputs_mask(groups))
    for p in (a, b):
        p.set_fields(d["close"], d["high"], d["low"], d["volume"])
    a.run_host(prm)
    _upload_and_run(pq, b, prm)
    for s in range(S):
        for name in (o for g in groups for o in OUTPUTS[g]):
            k = N.OUTPUT_NAMES.index(name)
            assert same(b.get_output(s, k), a.get_output(s, k)), (s, name)
    a.close()
    b.close()


# ---- 5. halts at chunk starts ------------------------------------------------------------------------------------------
NB_HALT, CHUNKS_HALT = 20_000, 8
L_HALT = geometry(NB_HALT, CHUNKS_HALT, 0)[0]                   # 2,528
HALTS = [  # (first, end) of a forward-filled halt, in bars; "3L" = the start of chunk 3
    ("3L-1200..3L+300", 3 * L_HALT - 1200, 3 * L_HALT + 300),
    ("3L-820..3L+300", 3 * L_HALT - 820, 3 * L_HALT + 300),
    ("3L-1200..3L-100", 3 * L_HALT - 1200, 3 * L_HALT - 100),
    ("3L-1200..3L-5", 3 * L_HALT - 1200, 3 * L_HALT - 5),
    ("3L-1200..3L-400", 3 * L_HALT - 1200, 3 * L_HALT - 400),
    ("3L-700..3L", 3 * L_HALT - 700, 3 * L_HALT),
    ("3L-600..3L", 3 * L_HALT - 600, 3 * L_HALT),
    ("3L+200..3L+1000 (output region only)", 3 * L_HALT + 200, 3 * L_HALT + 1000),
    ("300..1000 (chunk 0)", 300, 1000),
    ("end of the row", NB_HALT - 700, NB_HALT),
    ("no halt", 0, 0),
]
HALT_SETS = {"rsi-dm": ("rsi", "dm"), "rsi-dm-atr-natr-ema-trix": ("rsi", "dm", "atr", "natr", "ema", "trix"),
             "dm-atr-ema": ("dm", "atr", "ema")}
FILLS = ("close", "per-column")     # h = l = c = the last close; or each field keeps its own last value (prepare_sequential_data)


@pytest.mark.parametrize("path", ["run_host", "upload_run"])
@pytest.mark.parametrize("which", list(HALT_SETS))
def test_halts_at_chunk_starts(pq, which, path):
    groups = HALT_SETS[which]
    rows = [(fill, label, a, b) for fill in FILLS for label, a, b in HALTS]
    S = len(rows)
    d = synth.ohlcv(S, NB_HALT, seed=5)
    for s, (fill, _, a, b) in enumerate(rows):
        if b > a:                                       # a halt forward-filled onto the grid
            for f in ("close", "high", "low"):
                d[f][s, a:b] = d["close" if fill == "close" else f][s, a - 1]
            d["volume"][s, a:b] = 0.0
    prm = params(groups)
    W = pq.SplitPanel.required_warmup(prm)
    p = pq.SplitPanel(S, NB_HALT, chunks=CHUNKS_HALT, warmup=W, outputs_mask=outputs_mask(groups))
    assert p.chunk_bars == L_HALT
    p.set_fields(d["close"], d["high"], d["low"], d["volume"])
    if path == "run_host":
        p.run_host(prm)
    else:
        _upload_and_run(pq, p, prm)
    errs = []
    for s, (fill, label, _, _) in enumerate(rows):
        try:
            check_split(p, groups, prm, d, CHUNKS_HALT, W, expect_flat=True, symbols=[s])
        except AssertionError as e:
            errs.append(f"halt {label}, filled by {fill}: " + str(e).split("\nassert")[0].replace(f"symbol {s}: ", ""))
    p.close()
    assert not errs, f"W = {W}\n" + "\n".join(errs)
