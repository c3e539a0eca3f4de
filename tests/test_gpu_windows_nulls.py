"""Many-window panels (WindowPanel, BASELINE config 5) with halts, delistings, never-listed symbols and fields listed on
different rows, against the oracle's null rules and against the suite (Panel.compute) for the same single period, every
symbol and every bar, bit for bit in values and exactly in validity:
- KDJ: polars' positional rolling max / min with a full window (fastk null unless close is valid and the last k rows are valid
  in high and in low), the two calc_sma passes skip nulls, J = 3K - 2D where D is valid; flags do not kill KDJ;
- WILLR: all-null for a symbol flagged in close, high or low, else valid where close, high and low are, after p - 1 earlier
  bars with high and low valid;
- MIDPRICE / Donchian: all-null for a symbol flagged in high or low, else valid where high and low are, the expanding window
  counting only such bars;
- ATR: positional trange (previous row's close), calc_ema over the valid true ranges; flags do not kill ATR.
A field is flagged at its first null after its own first valid bar."""
import numpy as np
import pytest

import devread
import synth
import tolerances as T
from oracle import pqo

pytestmark = pytest.mark.gpu

F3 = ("close", "high", "low")
KDJ_ALL, EXT_A, EXT_B = (1, 5, 9, 33, 60, 250), (1, 5, 32, 33, 128), (250, 60)   # WMD 128 / 250: 16-bar segments, 33 / 60: 8
C5 = ((5, 9, 14, 60, 250), (5, 20, 55, 250), 14)


def _ok(S, N):
    return {f: np.ones((S, N), bool) for f in F3}


def _universe(S, N, seed=1):
    """One null pattern per symbol, cycling: none; close halted 3 bars (WILLR dies, MIDPRICE / Donchian live); all fields
    halted; one null in high; low halted 2 bars; delisted; never listed; listed late (leading nulls only); fields listed on
    different rows; high listed late only; a halt longer than every window; clustered close halts; nulls on the first and
    last bar of an 8-bar stage; a halt inside the first re-read segments of a two-level window."""
    rng = np.random.default_rng(seed)
    ok = _ok(S, N)
    for s in range(S):
        kind, t = s % 14, int(rng.integers(N // 8, N - N // 8))
        if kind == 1:
            ok["close"][s, t:t + 3] = False
        elif kind == 2:
            for f in F3: ok[f][s, t:t + 4] = False
        elif kind == 3:
            ok["high"][s, t] = False
        elif kind == 4:
            ok["low"][s, t:t + 2] = False
        elif kind == 5:
            for f in F3: ok[f][s, t:] = False
        elif kind == 6:
            for f in F3: ok[f][s] = False
        elif kind == 7:
            for f in F3: ok[f][s, :t] = False
        elif kind == 8:
            for f, a in zip(F3, (int(rng.integers(0, 40)), int(rng.integers(0, 40)), int(rng.integers(0, 40)))):
                ok[f][s, :a] = False
        elif kind == 9:
            ok["high"][s, :t] = False
        elif kind == 10:
            for f in F3: ok[f][s, N // 8:N // 8 + 300] = False
        elif kind == 11:
            for q in range(3):
                u = int(rng.integers(10, N - 10))
                ok["close"][s, u:u + 3] = False
        elif kind == 12:
            m = 8 * int(rng.integers(2, N // 8 - 2))
            ok["high"][s, m] = False
            ok["low"][s, m + 7] = False
        elif kind == 13:
            for f in F3: ok[f][s, 60 + 8:60 + 13] = False     # window 60: segment 1 of block 1, re-read while block 2 walks it
    return ok


def _set_panel(panel, d, ok, starts=None):
    S = d["close"].shape[0]
    for s in range(S):
        for f in F3:
            bits = None if ok[f][s].all() else np.packbits(ok[f][s].astype(np.uint8), bitorder="little")
            panel.set_column(s, f, d[f][s], validity=bits)
    if starts is not None:
        panel.set_fields(starts=starts)


def _windows(d, ok, kdj, ext, atr, starts=None, sk=3, sd=3, keep=False, **kw):
    from polars_quant_b200.windows import WindowPanel
    S, N = d["close"].shape
    wp = WindowPanel(S, N, kdj=kdj, ext=ext, atr=atr, slowk_period=sk, slowd_period=sd, **kw)
    _set_panel(wp.panel, d, ok, starts)
    res = {k: (v.copy(), m.copy()) for k, (v, m) in wp.compute().items()}
    if keep:
        return wp, res
    wp.close()
    return res


def _padded(n, a, ref):
    v, k = np.full(n, np.nan), np.zeros(n, bool)
    v[a:], k[a:] = ref
    return v, k


def expected(d, ok, s, kdj, ext, atr, sk=3, sd=3, flagged=None):
    """{line: (values, validity)} of symbol s under the null rules.  `ok` already holds the symbol's explicit start;
    `flagged` ({field: bool}) comes from the columns' own validity, which the intake flags before any start applies
    (default: from `ok`)."""
    n = d["close"].shape[1]
    c, h, l = (np.ascontiguousarray(d[f][s]) for f in F3)
    kc, kh, kl = (np.ascontiguousarray(ok[f][s]).astype(np.uint8) for f in F3)
    out = {}
    for k in kdj:
        K, D = pqo.stoch(h, l, c, k, sk, 0, sd, 0, kh, kl, kc)
        jok = K[1] & D[1]
        out["kdj_k_%d" % k], out["kdj_d_%d" % k] = K, D
        out["kdj_j_%d" % k] = (np.where(jok, 3.0 * K[0] - 2.0 * D[0], np.nan), jok)
    first = {f: (int(np.argmax(ok[f][s])) if ok[f][s].any() else None) for f in F3}
    if flagged is None:
        flagged = _flags(ok, s)
    hl = ok["high"][s] & ok["low"][s]
    a = int(np.argmax(hl)) if hl.any() else None
    none = (np.full(n, np.nan), np.zeros(n, bool))
    for p in ext:
        names = ["%s_%d" % (x, p) for x in ("willr", "midprice", "donchian_upper", "donchian_lower")]
        if a is None or flagged["high"] or flagged["low"]:
            for name in names: out[name] = none
            continue
        out[names[1]] = _padded(n, a, pqo.midprice(h[a:], l[a:], p))
        up, lo = pqo.donchian(h[a:], l[a:], p)
        out[names[2]], out[names[3]] = _padded(n, a, up), _padded(n, a, lo)
        if flagged["close"]:
            out[names[0]] = none
        else:
            # the window counts the bars from the first one with high and low valid; close must be valid at the bar itself
            wv, wk = _padded(n, a, pqo.willr(h[a:], l[a:], c[a:], p))
            wk = wk & ok["close"][s]
            out[names[0]] = (np.where(wk, wv, np.nan), wk)
    if atr:
        out["atr_%d" % atr] = pqo.atr(h, l, c, atr, kh, kl, kc)
    return out


def _flags(ok, s):
    """field -> a null after the field's first valid bar (the intake's flag)"""
    out = {}
    for f in F3:
        v = ok[f][s]
        out[f] = bool(v.any()) and not v[int(np.argmax(v)):].all()
    return out


def _folded(ok, starts):
    """the validity words' view: explicit starts folded into every field"""
    if starts is None:
        return ok
    f = {k: v.copy() for k, v in ok.items()}
    for s, a in enumerate(starts):
        for k in F3: f[k][s, :a] = False
    return f


def check_oracle(res, d, ok, kdj, ext, atr, starts=None, sk=3, sd=3, symbols=None, tag=""):
    raw, ok = ok, _folded(ok, starts)
    for s in (range(d["close"].shape[0]) if symbols is None else symbols):
        for name, (rv, rk) in expected(d, ok, s, kdj, ext, atr, sk, sd, _flags(raw, s)).items():
            nbad, msg = T.compare(name, res[name][0][s], res[name][1][s], rv, rk)
            assert nbad == 0, f"{tag} symbol {s}: {msg}"


def check_suite(res, d, ok, kdj, ext, atr, starts=None, sk=3, sd=3, tag=""):
    """Each line against Panel.compute with the same single period on the same columns (one suite run per KDJ / WMD
    window pair; the suite carries one period per indicator)."""
    import polars_quant_b200 as pq
    from polars_quant_b200 import _native as N
    S, n = d["close"].shape
    names = ("kdj_k", "kdj_d", "kdj_j", "willr", "midprice", "atr", "donchian_upper", "donchian_lower")
    om = sum(1 << N.OUTPUT_NAMES.index(x) for x in names)
    for i in range(max(len(kdj), len(ext), 1 if atr else 0)):
        ind, prm, lines = 0, {}, {}
        if i < len(kdj):
            ind |= N.IND["kdj"]
            prm.update(kdj_fastk=kdj[i], kdj_slowk=sk, kdj_slowd=sd)
            lines.update({"kdj_%s_%d" % (x, kdj[i]): "kdj_" + x for x in "kdj"})
        if i < len(ext):
            ind |= N.IND["willr"] | N.IND["midprice"] | N.IND_EXTRA["donchian"]
            prm.update(willr_period=ext[i], midprice_period=ext[i], donchian_period=ext[i])
            lines.update({"%s_%d" % (x, ext[i]): x for x in ("willr", "midprice", "donchian_upper", "donchian_lower")})
        if i == 0 and atr:
            ind |= N.IND["atr"]
            prm.update(atr_period=atr)
            lines["atr_%d" % atr] = "atr"
        panel = pq.Panel(S, n, outputs_mask=om)
        _set_panel(panel, d, ok, starts)
        panel.set_column(0, "volume", np.ones(n))
        for s in range(1, S):
            panel.set_column(s, "volume", np.ones(n))
        try:
            ref = panel.compute(N.default_params(indicators=ind, **prm))
        except N.PqbError:
            panel.close()
            continue                                   # (a period the suite's ring area does not take)
        for mine, theirs in lines.items():
            assert np.array_equal(res[mine][1], ref[theirs][1]), f"{tag} {mine}: validity differs from the suite's"
            assert T.same_bits(res[mine][0], ref[theirs][0]).all(), f"{tag} {mine}: values differ from the suite's"
        panel.close()


def test_every_window_kind_on_a_real_universe():
    """One-level and two-level KDJ / WMD windows and ATR 1 / 14 on a ragged 3-block panel of every null pattern."""
    S, N = 70, 700
    d = synth.ohlcv(S, N, seed=41)
    ok = _universe(S, N, seed=2)
    for kdj, ext, atr in ((KDJ_ALL, EXT_A, 14), ((), EXT_B, 1), ((250,), (33,), 0)):
        res = _windows(d, ok, kdj, ext, atr)
        check_oracle(res, d, ok, kdj, ext, atr, tag=f"{kdj} {ext} {atr}")
        check_suite(res, d, ok, kdj, ext, atr, tag=f"{kdj} {ext} {atr}")


def test_close_only_flag_keeps_midprice_and_donchian():
    S, N = 33, 300
    d = synth.ohlcv(S, N, seed=4)
    ok = _ok(S, N)
    ok["close"][3, 100:103] = False
    ok["close"][32, 299] = False                      # the ragged block's only symbol, flagged on the last bar
    res = _windows(d, ok, (9,), (5, 40), 14)
    for p in (5, 40):
        assert not res["willr_%d" % p][1][3].any() and not res["willr_%d" % p][1][32].any()
        assert res["midprice_%d" % p][1][3].all() and res["donchian_upper_%d" % p][1][32].all()
    check_oracle(res, d, ok, (9,), (5, 40), 14)
    check_suite(res, d, ok, (9,), (5, 40), 14)


def test_halts_at_stage_segment_and_window_edges():
    """Halts on the first and last bar of 8-bar stages, inside the segments a two-level window re-reads (windows 60 and
    128: 8- and 16-bar segments), across a block boundary, and longer than the window."""
    S, N = 40, 900
    d = synth.ohlcv(S, N, seed=9)
    ok = _ok(S, N)
    spots = [(0, 8, 1), (1, 15, 1), (2, 64, 3), (3, 120, 9), (4, 128 + 16, 16), (5, 255, 2), (6, 256, 1), (7, 300, 400),
             (8, 59, 2), (9, 60 * 3 + 8, 8), (10, 128 * 2 + 5, 20)]
    for s, t, ln in spots:
        for f in F3: ok[f][s, t:t + ln] = False
    for s, t, ln in spots:                            # the same spots in one field at a time
        ok["high"][s + 11, t:t + ln] = False
        ok["low"][s + 22, t + 1:t + 1 + ln] = False
    kdj, ext, atr = (33, 60, 250), (60, 128), 14
    res = _windows(d, ok, kdj, ext, atr)
    check_oracle(res, d, ok, kdj, ext, atr)
    check_suite(res, d, ok, kdj, ext, atr)


@pytest.mark.parametrize("sk,sd", ((1, 1), (1, 64), (64, 1), (64, 64)))
def test_kdj_smoothing_with_nulls(sk, sd):
    S, N = 40, 500
    d = synth.ohlcv(S, N, seed=sk + sd)
    ok = _universe(S, N, seed=sk * sd)
    res = _windows(d, ok, (9, 60), (), 0, sk=sk, sd=sd)
    check_oracle(res, d, ok, (9, 60), (), 0, sk=sk, sd=sd)
    check_suite(res, d, ok, (9, 60), (), 0, sk=sk, sd=sd)


def test_windows_longer_than_a_listed_history():
    S, N = 36, 400
    d = synth.ohlcv(S, N, seed=17)
    ok = _ok(S, N)
    for f in F3:
        ok[f][1, :N - 20] = False                      # listed 20 bars before the end
        ok[f][2, 30:] = False                          # delisted after 30 bars
        ok[f][3, :100] = False; ok[f][3, 150:] = False  # 50 listed bars
    ok["close"][4, :390] = False                       # close listed last, high / low from bar 0
    ok["high"][5, 200:] = False                        # delisted in high only
    res = _windows(d, ok, (60, 250), (60, 250), 14)
    check_oracle(res, d, ok, (60, 250), (60, 250), 14)
    check_suite(res, d, ok, (60, 250), (60, 250), 14)


def test_explicit_starts_with_nulls():
    S, N = 70, 600
    d = synth.ohlcv(S, N, seed=23)
    ok = _universe(S, N, seed=5)
    starts = np.zeros(S, dtype=np.int32)
    starts[[1, 2, 8, 13, 30, 33, 44, 66, 69]] = (20, 90, 7, 61, 250, 590, 599, 64, 600)
    # Flags come from the columns as given, before the start applies: a null before the start but after a field's first
    # valid bar still flags the field (symbol 30: a halt in every field and one more null in high, all before its start 250)
    ok["high"][30, 100] = False
    kdj, ext, atr = (5, 60), (5, 33), 14
    res = _windows(d, ok, kdj, ext, atr, starts=starts)
    check_oracle(res, d, ok, kdj, ext, atr, starts=starts)
    check_suite(res, d, ok, kdj, ext, atr, starts=starts)


def _same(a, b, name, rows):
    assert np.array_equal(a[name][1][rows], b[name][1][rows]), name
    assert a[name][0][rows].view(np.uint64).tobytes() == b[name][0][rows].view(np.uint64).tobytes(), name


def test_per_block_dispatch_and_the_return_to_the_plain_path():
    """Blocks without a flagged symbol are byte-identical to a run of the panel without those symbols' nulls; overwriting
    the flagged columns with clean ones brings back the plain path: same bits, same launch count."""
    S, N = 200, 500                                    # 7 blocks, the last one 8 symbols
    d = synth.ohlcv(S, N, seed=31)
    ok = _ok(S, N)
    for f in F3:
        ok[f][40, 200:203] = False                     # block 1
        ok[f][197, 400:] = False                       # block 6 (ragged), delisted
    ok["low"][140, 100] = False                        # block 4
    for f in F3:
        ok[f][70, :50] = False                         # block 2: leading nulls only (plain)
    kdj, ext, atr = C5
    wp, res = _windows(d, ok, kdj, ext, atr, keep=True)
    nl_null = wp.time_device(warmup=0, iters=1)[1]
    clean = _ok(S, N)
    for f in F3:
        clean[f][70, :50] = False
    wc, ref = _windows(d, clean, kdj, ext, atr, keep=True)
    nl_clean = wc.time_device(warmup=0, iters=1)[1]
    assert nl_clean == 2 and nl_null == 4, (nl_clean, nl_null)
    plain_rows = np.ones(S, bool)
    for b in (1, 4, 6):
        plain_rows[32 * b:32 * b + 32] = False
    for name in ref:
        _same(res, ref, name, plain_rows)
    check_oracle(res, d, ok, kdj, ext, atr, symbols=(40, 140, 197, 70, 33, 150))
    # overwrite the flagged columns with null-free ones: the panel returns to the plain kernel
    for s in (40, 140, 197):
        for f in F3:
            wp.panel.set_column(s, f, d[f][s])
    back = {k: (v.copy(), m.copy()) for k, (v, m) in wp.compute().items()}
    assert wp.time_device(warmup=0, iters=1)[1] == nl_clean
    for name in ref:
        _same(back, ref, name, slice(None))
    wp.close(); wc.close()


@pytest.mark.parametrize("env", ({"PQB_WIN_UNITS": "1"}, {"PQB_WIN_UNITS": "6", "PQB_WIN_STAGES": "4", "PQB_WIN_SMEM_MAX": "8"},
                                 {"PQB_WIN_STAGES": "3", "PQB_WIN_BLOCK_MAJOR": "1"}))
def test_planner_settings_give_the_default_plans_bits(monkeypatch, env):
    S, N = 70, 600
    d = synth.ohlcv(S, N, seed=61)
    ok = _universe(S, N, seed=7)
    for k in ("PQB_WIN_UNITS", "PQB_WIN_GROUPS", "PQB_WIN_PIPE", "PQB_WIN_SMEM_MAX", "PQB_WIN_STAGES", "PQB_WIN_BLOCK_MAJOR",
              "PQB_WIN_DEAL"):
        monkeypatch.delenv(k, raising=False)
    ref = _windows(d, ok, *C5)
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    res = _windows(d, ok, *C5)
    for name in ref:
        _same(res, ref, name, slice(None))
    check_oracle(res, d, ok, *C5, symbols=range(0, S, 5))


def test_time_device_then_compute():
    S, N = 70, 600
    d = synth.ohlcv(S, N, seed=71)
    ok = _universe(S, N, seed=8)
    wp, ref = _windows(d, ok, *C5, keep=True)
    ms, nl = wp.time_device(warmup=1, iters=3)
    assert ms > 0 and nl == 2                          # every block of this panel holds a flagged symbol
    res = wp.compute()
    for name in ref:
        _same(res, ref, name, slice(None))
    wp.close()


def test_config5_full_shape_with_halted_symbols():
    """10,000 x 5,040, config 5's windows, 1 % of the symbols halted for 3 bars in every field (one of them delisted, one
    flagged in close only), device-resident: the flagged symbols against the oracle, unflagged blocks against the clean run,
    read back from HBM."""
    import polars_quant_b200 as pq
    from polars_quant_b200.windows import WindowPanel
    S, N = 10_000, 5_040
    lib = pq._native.lib()
    kdj, ext, atr = C5
    wc = WindowPanel(S, N, kdj=kdj, ext=ext, atr=atr, host_staging=False)
    wc.fill_synthetic(seed=55, sigma=0.02)
    wc.run()
    wp = WindowPanel(S, N, kdj=kdj, ext=ext, atr=atr)
    wp.fill_synthetic(seed=55, sigma=0.02, to_host=True)
    halted = np.arange(7, S, 100)
    okrow = np.ones(N, bool)
    okrow[2000:2003] = False
    for i, s in enumerate(halted):
        s = int(s)
        row = okrow.copy()
        if i == 1:
            row[4000:] = False                         # delisted
        for f in F3:
            r = row if (i != 2 or f == "close") else np.ones(N, bool)   # symbol halted[2]: close only
            wp.panel.set_column(s, f, np.ascontiguousarray(wp.panel.host_field(f)[s]),
                                validity=np.packbits(r.astype(np.uint8), bitorder="little"))
    wp.panel.upload()
    wp.run()
    wp.panel.sync(); wc.panel.sync()
    assert wp.time_device(warmup=0, iters=1)[1] == 4
    nb, bp = wp.panel.tiled_shape()
    names = wp.names()
    flagged_blocks = sorted(set(int(s) // 32 for s in halted))

    def read(w, b):
        ns = min(32, S - b * 32)
        h_ = w.panel._h
        f = {name: devread.read_block(lib.pqb_panel_device_field(h_, k), b, bp, N)[:ns] for k, name in enumerate(F3)}
        outs = {names[k]: devread.read_block(lib.pqb_panel_device_output(h_, k), b, bp, N)[:ns] for k in names}
        oks = {names[k]: devread.read_validity_rows(lib.pqb_panel_device_validity(h_, k), b * 32, ns, w.panel.validity_pitch, N)
               for k in names}
        return f, outs, oks

    for b in flagged_blocks[:12] + [flagged_blocks[-1]]:
        f, outs, oks = read(wp, b)
        d = {k: v for k, v in f.items()}
        ok = {k: np.ones_like(v, dtype=bool) for k, v in f.items()}
        for i, s in enumerate(halted):
            if int(s) // 32 != b:
                continue
            row = okrow.copy()
            if i == 1:
                row[4000:] = False
            for k in F3:
                ok[k][int(s) % 32] = row if (i != 2 or k == "close") else True
        res = {name: (outs[name], oks[name]) for name in outs}
        check_oracle(res, d, ok, kdj, ext, atr, symbols=sorted(set([int(s) % 32 for s in halted if int(s) // 32 == b] + [0])),
                     tag=f"block {b}")
    unflagged = [b for b in range(nb) if b not in flagged_blocks]
    for b in unflagged[:3] + unflagged[len(unflagged) // 2:len(unflagged) // 2 + 2] + unflagged[-2:]:
        _, o1, k1 = read(wp, b)
        _, o2, k2 = read(wc, b)
        for name in o1:
            assert np.array_equal(k1[name], k2[name]), (b, name)
            assert o1[name].view(np.uint64).tobytes() == o2[name].view(np.uint64).tobytes(), (b, name)
    wp.close(); wc.close()
