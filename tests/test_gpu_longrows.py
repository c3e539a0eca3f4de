"""Long rows parallel along time (BASELINE config 3): K EMAs + MACD in one pass against the serial oracle, every symbol and
every bar: validity exact, the tile that holds a chain's seed bar and every tile before it bit-exact, later tiles within
the tolerance (rel 1e-10 / abs 1e-12 for the EMA lines; the MACD lines, differences of price-level EMAs that cross zero, add a
few ulp of the row's price level)."""
import numpy as np
import pytest

import devread
import synth
import tolerances as T
from oracle import pqo

pytestmark = pytest.mark.gpu
REL, ABS = 1e-10, 1e-12
ERR_INVALID, ERR_UNSUPPORTED, ERR_NULLS = -3, -4, -5
MACD_LINES = ("macd", "macd_signal", "macd_hist")
# MACD lines: |err| <= ABS + REL |ref| + MACD_ULPS * ulp(max |close| of the row).  Measured on a B200 (1,000 W power limit)
# by test_price_scale_bounds_the_macd_error_by_ulps_of_the_price_level (40 x 200,000, 1,024-bar tiles, price levels 1e-3 ..
# 1e5): at most 2.0 ulp at every level; the bound allows twice that.
MACD_ULPS = 4


def _close_enough(name, got, ref, ulp=0.0):
    """Validity exact; NaN where the oracle has NaN, the oracle's infinities; finite values within ABS + REL |ref| (+ ulp)."""
    (gv, gok), (rv, rok) = got, ref
    assert np.array_equal(gok, rok), f"{name}: validity differs at {np.argwhere(gok != rok)[:4].ravel().tolist()}"
    g, r = gv[rok], rv[rok]
    assert np.array_equal(np.isnan(g), np.isnan(r)), f"{name}: NaN differs at {np.argwhere(np.isnan(g) != np.isnan(r))[:4].ravel().tolist()}"
    fin = np.isfinite(r)
    assert T.same_bits(g[~fin], r[~fin]).all(), f"{name}: infinities differ"
    d = np.abs(g[fin] - r[fin])
    lim = ABS + REL * np.abs(r[fin]) + ulp
    if not (d <= lim).all():
        i = int(np.argmax(d - lim))
        raise AssertionError(f"{name}: max err {d.max():.3e} at {i}, allowed {lim[i]:.3e}")


def _check_all(res, close, periods, macd, tile):
    """Every symbol, every bar: within the tolerance, and bit for bit through the tile that holds each seed bar (through
    the whole row when one tile holds it)."""
    for s in range(close.shape[0]):
        for p in periods:
            got = (res["ema_%d" % p][0][s], res["ema_%d" % p][1][s])
            ref = pqo.ema(close[s], p)
            _close_enough(f"symbol {s} ema({p}) tile {tile}", got, ref)
            first = max(tile, (p - 1) // tile * tile + tile)          # through the tile that holds the seed bar: the reference itself
            nbad, msg = T.compare(f"symbol {s} ema({p})", got[0][:first], got[1][:first], ref[0][:first], ref[1][:first])
            assert nbad == 0, msg
        if macd:
            for name, ref in zip(MACD_LINES, pqo.macd(close[s], *macd)):
                got = (res[name][0][s], res[name][1][s])
                _close_enough(f"symbol {s} {name}{macd} tile {tile}", got, ref)
                nbad, msg = T.compare(f"symbol {s} {name}{macd}", got[0][:tile], got[1][:tile], ref[0][:tile], ref[1][:tile])
                assert nbad == 0, msg


def _copy(res):
    return {k: (v.copy(), ok.copy()) for k, (v, ok) in res.items()}


def test_ema_set_and_macd_against_the_serial_oracle():
    from polars_quant_b200.longrows import LongPanel
    S, NB = 70, 30_000
    d = synth.ohlcv(S, NB, seed=3, sigma=0.0005)
    for tile, periods, macd in ((256, (12, 26, 200, 5000), (12, 26, 9)), (1024, (5, 300), (3, 10, 16)), (512, (30,), None),
                                (64, (), (12, 26, 9))):
        lp = LongPanel(S, NB, ema_periods=periods, macd=macd, tile_bars=tile)
        lp.panel.set_fields(close=d["close"])
        _check_all(lp.compute(), d["close"], periods, macd, tile)
        lp.close()


@pytest.mark.parametrize("n_bars", (1, 2, 15, 16, 17, 63, 64, 65, 1000))
def test_one_tile_is_the_reference_bit_for_bit(n_bars):
    """tile_bars >= n_bars: the whole row is tile 0, the reference's own computation -- including rows shorter than the
    MACD's slow period (dif all null, the signal line an EMA of the zero-filled dif), fast > slow, and period 1."""
    from polars_quant_b200.longrows import LongPanel
    S = 33
    d = synth.ohlcv(S, n_bars, seed=40 + n_bars, sigma=0.01)
    tile = max(64, n_bars)
    periods = (1, 2, 5, 12, 64)
    for macd in ((12, 26, 9), (26, 12, 9), (1, 2, 1)):
        lp = LongPanel(S, n_bars, ema_periods=periods, macd=macd, tile_bars=tile)
        lp.panel.set_fields(close=d["close"])
        res = lp.compute()
        for s in range(S):
            refs = {"ema_%d" % p: pqo.ema(d["close"][s], p) for p in periods}
            refs.update(zip(MACD_LINES, pqo.macd(d["close"][s], *macd)))
            for name, (rv, rk) in refs.items():
                nbad, msg = T.compare(name, res[name][0][s], res[name][1][s], rv, rk)
                assert nbad == 0, f"n_bars {n_bars} macd {macd} symbol {s}: {msg}"
        lp.close()


@pytest.mark.parametrize("n_bars", (127, 128, 129, 255, 256, 257))
def test_seed_bars_on_and_around_tile_edges(n_bars):
    """L = 64: seed bars p - 1 at L - 2, L - 1, L, L + 1, 2L - 1, 2L and 3L + 5 (lr_carry_kernel switches from a zero start
    to the seed exactly at the seed's tile), one valid bar (p = n_bars) and none (p = n_bars + 1)."""
    from polars_quant_b200.longrows import LongPanel
    L, S = 64, 40
    d = synth.ohlcv(S, n_bars, seed=n_bars, sigma=0.001)
    for periods, macd in (((63, 64, 65, 66), (12, 26, 9)), ((128, 129, 198), None), ((n_bars, n_bars + 1), (12, 26, 9))):
        lp = LongPanel(S, n_bars, ema_periods=periods, macd=macd, tile_bars=L)
        lp.panel.set_fields(close=d["close"])
        _check_all(lp.compute(), d["close"], periods, macd, L)
        lp.close()


@pytest.mark.parametrize("S", (70, 33))
def test_seven_and_eight_chains(S):
    """lr_local_kernel has straight-line paths for 1 - 6 chains; with 7 or 8 (LR_MAX_CH) the interior tiles take the
    general path.  7 EMA outputs, two of them sharing the MACD's chains: 7 chains; 6 EMAs and a distinct MACD: 8."""
    from polars_quant_b200.longrows import LongPanel
    NB, tile = 5000, 256
    d = synth.ohlcv(S, NB, seed=S, sigma=0.0005)
    for periods, macd in (((12, 26, 5, 50, 100, 200, 300), (12, 26, 9)), ((5, 50, 100, 200, 300, 7), (12, 26, 9))):
        lp = LongPanel(S, NB, ema_periods=periods, macd=macd, tile_bars=tile)
        lp.panel.set_fields(close=d["close"])
        _check_all(lp.compute(), d["close"], periods, macd, tile)
        lp.close()


def test_short_rows_and_guards():
    from polars_quant_b200.longrows import LongPanel
    from polars_quant_b200 import _native as N
    d = synth.ohlcv(3, 100, seed=4)
    lp = LongPanel(3, 100, ema_periods=(30, 200), macd=(12, 26, 9), tile_bars=64)
    lp.panel.set_fields(close=d["close"])
    res = lp.compute()
    assert not res["ema_200"][1].any()                                     # n < p: all null (overlap.rs:663)
    _check_all(res, d["close"], (30, 200), (12, 26, 9), 64)
    lp.close()
    with pytest.raises(N.PqbError) as e:
        LongPanel(3, 100, ema_periods=(), macd=None)
    assert e.value.code == ERR_INVALID
    with pytest.raises(N.PqbError) as e:
        LongPanel(3, 100, ema_periods=(2, 3, 4, 5, 6, 7, 8, 9), macd=None)   # 8 EMA outputs (LR_MAX_EMA = 7)
    assert e.value.code == ERR_INVALID
    lp = LongPanel(3, 5000, ema_periods=(10,), macd=(12, 2000, 9), tile_bars=256)
    lp.panel.set_fields(close=np.ones((3, 5000)))
    lp.panel.upload()
    with pytest.raises(N.PqbError, match="first time tile") as e:
        lp.run()
    assert e.value.code == ERR_UNSUPPORTED
    lp.close()
    x = d["close"][:, :100]
    for periods, macd in (((5, 50, 100, 200, 300, 7, 8), (12, 26, 9)),   # 9 distinct chains (LR_MAX_CH = 8)
                          ((10, 10), None),                               # the same EMA period twice
                          ((10,), (12, 12, 9)),                           # fast == slow
                          ((0,), None), ((10,), (0, 26, 9)), ((10,), (12, 26, 0))):
        lp = LongPanel(3, 100, ema_periods=periods, macd=macd, tile_bars=64)
        lp.panel.set_fields(close=x)
        lp.panel.upload()
        with pytest.raises(N.PqbError) as e:
            lp.run()
        assert e.value.code == ERR_UNSUPPORTED, (periods, macd, str(e.value))
        lp.close()
    # null-bearing columns are the time-split / serial path's job: starts, and an Arrow null in close
    lp = LongPanel(3, 100, ema_periods=(10,), macd=(12, 26, 9), tile_bars=64)
    lp.panel.set_fields(close=x, starts=np.array([0, 5, 0], dtype=np.int32))
    with pytest.raises(N.PqbError) as e:
        lp.compute()
    assert e.value.code == ERR_NULLS
    lp.close()
    lp = LongPanel(3, 100, ema_periods=(10,), macd=(12, 26, 9), tile_bars=64)
    lp.panel.set_fields(close=x)
    bits = np.packbits(np.arange(100) != 40, bitorder="little")
    lp.panel.set_column(1, "close", x[1], bits)
    with pytest.raises(N.PqbError) as e:
        lp.compute()
    assert e.value.code == ERR_NULLS
    lp.close()


def test_nan_and_inf_close_on_tile_edges():
    """NaN / +inf at a tile's first bar, last bar and inside it, in tile 0, in the tile that holds EMA(200)'s seed bar and
    in interior tiles (the straight-line path; period 1 has A = 0, where the carry computes fma(0, inf, B)): NaN positions
    and validity equal the oracle's, finite values within the tolerance."""
    from polars_quant_b200.longrows import LongPanel
    L, S, NB = 64, 40, 520
    d = synth.ohlcv(S, NB, seed=12, sigma=0.001)
    close = d["close"].copy()
    bars = (0, 63, 64, 100, 127, 192, 199, 255, 256, 300, 319, 320, 383, 511, 512, 519)
    for s in range(2 * len(bars)):
        close[s, bars[s % len(bars)]] = np.nan if s < len(bars) else np.inf
    close[2 * len(bars), [70, 330]] = np.inf, np.nan
    periods, macd = (1, 2, 12, 200), (12, 26, 9)
    lp = LongPanel(S, NB, ema_periods=periods, macd=macd, tile_bars=L)
    lp.panel.set_fields(close=close)
    _check_all(lp.compute(), close, periods, macd, L)
    lp.close()


def test_reruns_and_new_closes_give_the_same_bits():
    from polars_quant_b200.longrows import LongPanel
    S, NB, tile = 40, 3000, 256
    periods, macd = (12, 200), (12, 26, 9)
    a = synth.ohlcv(S, NB, seed=21, sigma=0.0005)["close"]
    b = synth.ohlcv(S, NB, seed=22, sigma=0.0005)["close"]

    def same(x, y):
        for k in x:
            assert np.array_equal(x[k][1], y[k][1]), k
            assert T.same_bits(x[k][0], y[k][0]).all(), k

    lp = LongPanel(S, NB, ema_periods=periods, macd=macd, tile_bars=tile)
    lp.panel.set_fields(close=a)
    first = _copy(lp.compute())
    same(first, lp.compute())
    _check_all(first, a, periods, macd, tile)
    lp.panel.set_fields(close=b)
    second = _copy(lp.compute())
    fresh = LongPanel(S, NB, ema_periods=periods, macd=macd, tile_bars=tile)
    fresh.panel.set_fields(close=b)
    same(second, fresh.compute())
    fresh.close()
    lp.time_device(warmup=1, iters=2)
    same(second, lp.compute())
    lp.close()


def test_price_scale_bounds_the_macd_error_by_ulps_of_the_price_level():
    """close = level x a synthetic path, level 1e-3 .. 1e5.  Tiles after the first start from a carried state a few ulp off
    the serial one.  The EMA lines stay within rel 1e-10 / abs 1e-12 at every level; the MACD lines are differences of
    price-level EMAs that cross zero, so their error is bounded by ulps of the price level, not by abs 1e-12."""
    from polars_quant_b200.longrows import LongPanel
    S, NB, tile = 40, 200_000, 1024
    periods, macd = (12, 26, 200, 5000), (12, 26, 9)
    path = synth.ohlcv(S, NB, seed=3, sigma=0.0005)["close"] / 100.0
    lp = LongPanel(S, NB, ema_periods=periods, macd=macd, tile_bars=tile)
    worst, over = {}, {}
    for level in (1e-3, 1.0, 1e2, 1e4, 1e5):
        close = path * level
        lp.panel.set_fields(close=close)
        res = lp.compute()
        k, n_over = 0.0, 0
        for s in range(S):
            for p in periods:
                _close_enough(f"level {level} symbol {s} ema({p})", (res["ema_%d" % p][0][s], res["ema_%d" % p][1][s]),
                              pqo.ema(close[s], p))
            ulp = np.spacing(np.abs(close[s]).max())
            for name, (rv, rk) in zip(MACD_LINES, pqo.macd(close[s], *macd)):
                got = (res[name][0][s], res[name][1][s])
                d = np.abs(got[0][rk] - rv[rk])
                k = max(k, float((d / ulp).max()))
                n_over += int((d > ABS + REL * np.abs(rv[rk])).sum())
                if level == 1e2:
                    _close_enough(f"level {level} symbol {s} {name}", got, (rv, rk))          # the plain abs 1e-12 holds here
                _close_enough(f"level {level} symbol {s} {name}", got, (rv, rk), MACD_ULPS * ulp)
        worst[level], over[level] = k, n_over
    print("MACD lines: max |err| / ulp(max |close| of the row) by price level:", worst)
    print("MACD values outside abs 1e-12 / rel 1e-10 by price level:", over)
    lp.close()


def test_config3_full_shape_against_the_oracle():
    """500 symbols x 1,000,000 bars, EMA(12, 26, 200, 5000) + MACD(12, 26, 9), device-resident synthetic minute bars: two
    symbol blocks are read back from HBM and compared with the serial oracle over the whole million bars."""
    import polars_quant_b200 as pq
    from polars_quant_b200.longrows import LongPanel
    S, NB = 500, 1_000_000
    lib = pq._native.lib()
    lp = LongPanel(S, NB, ema_periods=(12, 26, 200, 5000), macd=(12, 26, 9), host_staging=False)
    lp.fill_synthetic(seed=3, sigma=0.0005)
    lp.run()
    lp.panel.sync()
    nb, bp = lp.panel.tiled_shape()
    h = lp.panel._h
    names = lp.names()
    for b in (0, nb - 1):
        ns = min(32, S - b * 32)
        close = devread.read_block(lib.pqb_panel_device_field(h, 0), b, bp, NB)[:ns]
        outs = {k: devread.read_block(lib.pqb_panel_device_output(h, k), b, bp, NB)[:ns] for k in names}
        oks = {k: devread.read_validity_rows(lib.pqb_panel_device_validity(h, k), b * 32, ns, lp.panel.validity_pitch, NB) for k in names}
        for s in (0, ns // 2, ns - 1):
            refs = {0: pqo.ema(close[s], 12), 1: pqo.ema(close[s], 26), 2: pqo.ema(close[s], 200), 3: pqo.ema(close[s], 5000)}
            refs.update(dict(zip((7, 8, 9), pqo.macd(close[s], 12, 26, 9))))
            for k, ref in refs.items():
                _close_enough(f"block {b} symbol {s} {names[k]}", (outs[k][s], oks[k][s]), ref)
    lp.close()
