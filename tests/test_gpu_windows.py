"""Many rolling windows in one launch (BASELINE config 5) against the oracle: every value and validity bit identical to
the per-window reference calls (STOCH / KDJ momentum.py:178-186 + D3, willr momentum.rs:630, midprice overlap.rs:281,
Donchian lines D3, atr volatility.rs:18)."""
import numpy as np
import pytest

import devread
import synth
import tolerances as T
from oracle import pqo

pytestmark = pytest.mark.gpu


ERR_INVALID, ERR_UNSUPPORTED = -3, -4
C5 = ((5, 9, 14, 60, 250), (5, 20, 55, 250), 14)                 # config 5's windows: KDJ, WILLR / MIDPRICE / Donchian, ATR


def _refs(h, l, c, kdj, ext, atr, sk=3, sd=3):
    out = {}
    for k in kdj:
        K, D, J = pqo.kdj(h, l, c, k, sk, sd)
        out["kdj_k_%d" % k], out["kdj_d_%d" % k], out["kdj_j_%d" % k] = K, D, J
    for p in ext:
        out["willr_%d" % p] = pqo.willr(h, l, c, p)
        out["midprice_%d" % p] = pqo.midprice(h, l, p)
        up, lo = pqo.donchian(h, l, p)
        out["donchian_upper_%d" % p], out["donchian_lower_%d" % p] = up, lo
    if atr:
        out["atr_%d" % atr] = pqo.atr(h, l, c, atr)
    return out


def _check_all(res, d, starts, kdj, ext, atr, sk=3, sd=3, tag=""):
    """Every symbol and every bar against the oracle run on the symbol's listed bars, bit for bit; validity exact."""
    S, N = d["close"].shape
    for s in range(S):
        a = int(starts[s]) if starts is not None else 0
        refs = _refs(d["high"][s, a:], d["low"][s, a:], d["close"][s, a:], kdj, ext, atr, sk, sd)
        for name, (rv, rk) in refs.items():
            fv = np.full(N, np.nan); fk = np.zeros(N, bool)
            fv[a:], fk[a:] = rv, rk
            nbad, msg = T.compare(name, res[name][0][s], res[name][1][s], fv, fk)
            assert nbad == 0, f"{tag} symbol {s} (start {a}): {msg}"


def _run(S, N, d, starts, kdj, ext, atr, **kw):
    from polars_quant_b200.windows import WindowPanel
    wp = WindowPanel(S, N, kdj=kdj, ext=ext, atr=atr, **kw)
    wp.panel.set_fields(close=d["close"], high=d["high"], low=d["low"], starts=starts)
    res = {k: (v.copy(), ok.copy()) for k, (v, ok) in wp.compute().items()}
    wp.close()
    return res


def test_window_suite_small_panels_and_listing_dates():
    from polars_quant_b200.windows import WindowPanel
    S, N = 75, 900
    d = synth.ohlcv(S, N, seed=21)
    kdj, ext, atr = (5, 9, 14, 60, 250), (5, 20, 55, 250), 14
    wp = WindowPanel(S, N, kdj=kdj, ext=ext, atr=atr)
    starts = np.zeros(S, dtype=np.int32)
    starts[[3, 40, 74]] = (17, 300, 640)
    wp.panel.set_fields(close=d["close"], high=d["high"], low=d["low"], starts=starts)
    res = wp.compute()
    assert len(res) == 15 + 16 + 1
    _check_all(res, d, starts, kdj, ext, atr)
    wp.close()
    # other shapes of the unit dealing: one window, no ATR, windows on both sides of the shared / global limit
    for kdj, ext, atr in (((9,), (), 0), ((), (64, 65), 7), ((3, 100), (2,), 0), ((33, 129), (40, 128, 499), 3), ((600,), (32, 33, 501), 0)):
        wp = WindowPanel(40, 500, kdj=kdj, ext=ext, atr=atr)
        wp.panel.set_fields(close=d["close"][:40, :500], high=d["high"][:40, :500], low=d["low"][:40, :500])
        res = wp.compute()
        _check_all(res, {k: d[k][:40, :500] for k in ("close", "high", "low")}, None, kdj, ext, atr, tag=f"{kdj} {ext} {atr}")
        wp.close()


@pytest.mark.parametrize("sk,sd", ((1, 1), (1, 3), (3, 1), (2, 5), (5, 2), (64, 1), (64, 64)))
def test_kdj_smoothing_periods(sk, sd):
    """KDJ's two calc_sma passes at smoothing periods 1 .. 64, on a one-level (9) and a two-level (60) window, with
    listing dates."""
    S, N = 40, 400
    d = synth.ohlcv(S, N, seed=sk * 100 + sd)
    starts = np.zeros(S, dtype=np.int32)
    starts[[1, 17, 33, 39]] = (3, 59, 200, 330)
    _check_all(_run(S, N, d, starts, (9, 60), (), 0, slowk_period=sk, slowd_period=sd), d, starts, (9, 60), (), 0, sk, sd)


def test_kdj_smoothing_periods_out_of_range_are_refused():
    from polars_quant_b200 import _native as N
    from polars_quant_b200.windows import WindowPanel
    for sk, sd in ((0, 3), (3, 0), (65, 3), (3, 65)):
        with pytest.raises(N.PqbError) as e:
            WindowPanel(8, 100, kdj=(9,), ext=(), atr=0, slowk_period=sk, slowd_period=sd)
        assert e.value.code == ERR_UNSUPPORTED, (sk, sd)


def test_every_unit_at_once_and_windows_of_one_bar():
    """12 units (W_MAX_TOTAL): six KDJ windows, five WILLR / MIDPRICE / Donchian windows and ATR, windows of one bar
    included; a seventh KDJ window is refused."""
    from polars_quant_b200 import _native as N
    from polars_quant_b200.windows import WindowPanel
    S, N_ = 70, 700
    d = synth.ohlcv(S, N_, seed=12)
    starts = np.zeros(S, dtype=np.int32)
    starts[[5, 31, 32, 69]] = (1, 130, 250, 699)
    kdj, ext, atr = (1, 5, 32, 33, 128, 250), (1, 31, 32, 33, 129), 1
    res = _run(S, N_, d, starts, kdj, ext, atr)
    assert len(res) == 3 * 6 + 4 * 5 + 1
    _check_all(res, d, starts, kdj, ext, atr)
    with pytest.raises(N.PqbError) as e:
        WindowPanel(S, N_, kdj=(1, 5, 32, 33, 128, 250, 7), ext=ext, atr=atr)
    assert e.value.code == ERR_INVALID
    with pytest.raises(N.PqbError) as e:
        WindowPanel(S, N_, kdj=kdj, ext=(1, 31, 32, 33, 129, 7), atr=atr)
    assert e.value.code == ERR_INVALID


@pytest.mark.parametrize("n_bars", (1, 7, 8, 9, 31, 33))
def test_short_histories(n_bars):
    """Panels shorter than most windows; symbols listed on the last bar and never listed (start = n_bars)."""
    S = 40
    d = synth.ohlcv(S, n_bars, seed=n_bars)
    starts = np.zeros(S, dtype=np.int32)
    starts[[2, 20, 33]] = n_bars - 1
    starts[[3, 34, 39]] = n_bars
    if n_bars > 4:
        starts[[4, 35]] = (n_bars // 2, 3)
    _check_all(_run(S, n_bars, d, starts, *C5), d, starts, *C5, tag=f"n_bars {n_bars}")


def test_listing_dates_around_a_two_level_window():
    """Window 60 (two-level, 8-bar segments, blocks of 60 bars aligned to absolute time): listed at p - 1, p, p + 1, on
    segment boundaries of the first and second block, and too late for a whole window."""
    S, N = 40, 400
    d = synth.ohlcv(S, N, seed=60)
    starts = np.zeros(S, dtype=np.int32)
    starts[1:12] = (59, 60, 61, 8, 16, 56, 64, 68, 120, 128, 350)
    kdj, ext, atr = (60,), (60,), 0
    _check_all(_run(S, N, d, starts, kdj, ext, atr), d, starts, kdj, ext, atr)


_KNOBS = ("PQB_WIN_UNITS", "PQB_WIN_GROUPS", "PQB_WIN_PIPE", "PQB_WIN_SMEM_MAX", "PQB_WIN_STAGES", "PQB_WIN_BLOCK_MAJOR",
          "PQB_WIN_DEAL", "PQB_WIN_RELAXED_WAIT", "PQB_WIN_VERBOSE")


@pytest.fixture(scope="module")
def ragged_c5():
    """Config 5's windows on a small ragged panel (3 symbol blocks, the last one 6 symbols) with listing dates, under the
    default plan."""
    S, N = 70, 700
    d = synth.ohlcv(S, N, seed=505)
    starts = np.zeros(S, dtype=np.int32)
    starts[[1, 30, 33, 64, 69]] = (7, 61, 250, 499, 690)
    with pytest.MonkeyPatch.context() as mp:
        for k in _KNOBS:
            mp.delenv(k, raising=False)
        res = _run(S, N, d, starts, *C5)
    _check_all(res, d, starts, *C5, tag="default plan")
    return S, N, d, starts, res


@pytest.mark.parametrize("env,expect", [({"PQB_WIN_UNITS": str(u)}, ["groups of <= %d," % u]) for u in range(1, 7)] + [
    ({"PQB_WIN_GROUPS": "10"}, ["10 units in 10 groups"]),
    ({"PQB_WIN_GROUPS": "12"}, ["10 units in 10 groups"]),          # more groups than units: clamped to one unit per group
    ({"PQB_WIN_UNITS": "3", "PQB_WIN_GROUPS": "5"}, ["10 units in 5 groups of <= 3,"]),
] + [({"PQB_WIN_PIPE": str(m)}, ["pipe mask %d," % m]) for m in range(4)] + [
    ({"PQB_WIN_SMEM_MAX": "16"}, ["one-level windows <= 16 bars"]),
    ({"PQB_WIN_SMEM_MAX": "8"}, ["one-level windows <= 8 bars"]),
    ({"PQB_WIN_SMEM_MAX": "4"}, ["one-level windows <= 8 bars"]),  # below 8: clamped (Ext2 needs two segments per block)
    ({"PQB_WIN_STAGES": "3"}, ["; 3 stages,"]),
    ({"PQB_WIN_STAGES": "4"}, ["; 4 stages,"]),
    ({"PQB_WIN_BLOCK_MAJOR": "1"}, ["block-major CTAs"]),
    ({"PQB_WIN_DEAL": "0"}, ["dealt by cost"]),
    ({"PQB_WIN_UNITS": "6", "PQB_WIN_SMEM_MAX": "8", "PQB_WIN_STAGES": "4", "PQB_WIN_PIPE": "0", "PQB_WIN_BLOCK_MAJOR": "1"},
     ["groups of <= 6,", "one-level windows <= 8 bars", "; 4 stages,", "pipe mask 0,", "block-major CTAs"]),
])
def test_every_plan_and_build_gives_the_same_bits(ragged_c5, monkeypatch, capfd, env, expect):
    """The planner's debug knobs (read by pqb_windows_create) reach the <192, 2> build (5 - 6 units per CTA), unpiped
    units, two-level arrays for windows of 9 - 32 bars, rings of 3 - 4 stages, block-major CTA order and cost dealing:
    every plan gives the default plan's bits, which are the oracle's.  The plan line proves that each knob took effect."""
    import re
    from polars_quant_b200.windows import WindowPanel
    S, N, d, starts, ref = ragged_c5
    for k in _KNOBS:
        monkeypatch.delenv(k, raising=False)
    monkeypatch.setenv("PQB_WIN_VERBOSE", "1")
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    capfd.readouterr()
    wp = WindowPanel(S, N, kdj=C5[0], ext=C5[1], atr=C5[2])
    line = [x for x in capfd.readouterr().err.splitlines() if x.startswith("[pqb windows]")][-1]
    for e in expect:
        assert e in line, line
    m = re.search(r"(\d+) units in (\d+) groups of <= (\d+), (\d+) threads per CTA", line)
    n_units, groups, per, threads = (int(x) for x in m.groups())
    assert n_units == 10 and groups <= n_units and -(-n_units // groups) <= per and threads <= 32 * per, line
    if "PQB_WIN_UNITS" in env and int(env["PQB_WIN_UNITS"]) >= 5:
        assert threads in (160, 192), line                             # the <192, 2> build
    if env.get("PQB_WIN_SMEM_MAX") == "4":                            # the clamped plan is the plan at 8
        monkeypatch.setenv("PQB_WIN_SMEM_MAX", "8")
        WindowPanel(S, N, kdj=C5[0], ext=C5[1], atr=C5[2]).close()
        line8 = [x for x in capfd.readouterr().err.splitlines() if x.startswith("[pqb windows]")][-1]
        assert line8 == line, (line, line8)
    wp.panel.set_fields(close=d["close"], high=d["high"], low=d["low"], starts=starts)
    res = wp.compute()
    for name, (rv, rk) in ref.items():
        assert np.array_equal(res[name][1], rk), f"{env}: {name} validity differs from the default plan's"
        assert T.same_bits(res[name][0], rv).all(), f"{env}: {name} differs from the default plan's bits"
    wp.close()


def test_config5_full_shape_against_the_oracle():
    """10,000 x 5,040, KDJ(5, 9, 14, 60, 250) + WILLR / MIDPRICE / Donchian(5, 20, 55, 250) + ATR(14), device-resident:
    symbol blocks across the grid are read back from HBM and compared with the oracle bit for bit."""
    import polars_quant_b200 as pq
    from polars_quant_b200.windows import WindowPanel
    S, N = 10_000, 5_040
    lib = pq._native.lib()
    kdj, ext, atr = (5, 9, 14, 60, 250), (5, 20, 55, 250), 14
    wp = WindowPanel(S, N, kdj=kdj, ext=ext, atr=atr, host_staging=False)
    wp.fill_synthetic(seed=55, sigma=0.02)
    wp.run()
    wp.panel.sync()
    nb, bp = wp.panel.tiled_shape()
    h_ = wp.panel._h
    names = wp.names()
    for b in (0, 1, 147, 148, 200, nb - 1):
        ns = min(32, S - b * 32)
        c, h, l = (devread.read_block(lib.pqb_panel_device_field(h_, f), b, bp, N)[:ns] for f in (0, 1, 2))
        outs = {k: devread.read_block(lib.pqb_panel_device_output(h_, k), b, bp, N)[:ns] for k in names}
        oks = {k: devread.read_validity_rows(lib.pqb_panel_device_validity(h_, k), b * 32, ns, wp.panel.validity_pitch, N) for k in names}
        for s in (0, ns - 1):
            refs = _refs(h[s], l[s], c[s], kdj, ext, atr)
            for k, name in names.items():
                nbad, msg = T.compare(name, outs[k][s], oks[k][s], refs[name][0], refs[name][1])
                assert nbad == 0, f"block {b} symbol {s}: {msg}"
    wp.close()


def test_long_windows_ignore_nan_highs_and_lows_like_the_reference():
    """The two-level window extremes (windows > 32) fold with the reference's f64::max / f64::min semantics (momentum.rs:644-650:
    a NaN value is ignored), exactly like the one-level ones: willr with NaN highs and lows.  (midprice and the Donchian
    lines follow other NaN rules, documented divergences: DESIGN.md section 5.)"""
    from polars_quant_b200.windows import WindowPanel
    S, N = 33, 700
    d = synth.ohlcv(S, N, seed=77)
    h, l, c = d["high"].copy(), d["low"].copy(), d["close"].copy()
    rng = np.random.default_rng(5)
    for s in range(S):
        idx = rng.choice(N, size=25, replace=False)
        h[s, idx[:12]] = np.nan
        l[s, idx[12:]] = np.nan
    h[7, 100:420] = np.nan                      # longer than every window but one: whole windows without a comparable value
    kdj, ext, atr = (), (20, 60, 250), 0
    wp = WindowPanel(S, N, kdj=kdj, ext=ext, atr=atr)
    wp.panel.set_fields(close=c, high=h, low=l)
    res = wp.compute()
    for s in (0, 7, 32):
        for p in ext:
            rv, rk = pqo.willr(h[s], l[s], c[s], p)
            nbad, msg = T.compare("willr_%d" % p, res["willr_%d" % p][0][s], res["willr_%d" % p][1][s], rv, rk)
            assert nbad == 0, f"symbol {s}: {msg}"
    wp.close()
