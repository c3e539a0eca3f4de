"""Live screens at the benchmark shape: prime a 50,000 x 5,040 synthetic history twice -- a live panel without a screen
and one with the default screen (crossover signals, SMA(10, 20) cross, info) -- and push k new random-walk bars per
symbol (k = 1, 8, 64) into both, alternating, with a cold L2 before every timed push.  Beside it, the whole-panel way to
the same answers on a recomputed 5,041-bar panel: the suite, pqb_signals_time, pqb_ma_cross_run and pqb_panel_info.
Prints one JSON line.

    python scripts/bench_live_screen.py [--symbols 50000] [--bars 5040] [--reps 20] [--out file.json]

device_ms: CUDA events of pqb_live_push (pack of the new rows .. the last screen kernel, no PCIe);
e2e_ms: host clock around pqb_live_push (host validation, H2D, kernels, D2H into pinned result rows)."""
import argparse
import ctypes as C
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

import polars_quant_b200 as pq                      # noqa: E402
from polars_quant_b200 import _native as N          # noqa: E402


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = (x.strip() for x in q.split(","))
        return name, power
    except Exception as ex:                          # (reported, not guessed)
        return "unknown (%s)" % ex, "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--symbols", type=int, default=50000)
    ap.add_argument("--bars", type=int, default=5040)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    S, T = a.symbols, a.bars
    eng, L = pq.get_engine(0), N.lib()
    params = N.default_params()

    hist = pq.Panel(S, T, outputs_mask=0, host_staging=False)
    hist.fill_synthetic(seed=0xC0FFEE, sigma=0.02)
    lives, prime_ms = {}, {}
    for name, screen in (("plain", None), ("screen", dict(ma_cross=("sma", 10, 20), info=True))):
        t0 = time.perf_counter()
        lives[name] = pq.LivePanel(hist, params, None, 64, screen=screen)     # (create ends with a device synchronise)
        prime_ms[name] = (time.perf_counter() - t0) * 1e3
    hist.close()

    rng = np.random.default_rng(1)
    last = np.full(S, 100.0)

    def bars(k):
        nonlocal last
        c = last * np.exp(np.cumsum(0.02 * rng.standard_normal((k, S)), axis=0))
        o = np.vstack([last[None, :], c[:-1]])
        h = np.maximum(o, c) * (1.0 + np.abs(0.01 * rng.standard_normal((k, S))))
        lo = np.minimum(o, c) * (1.0 - np.abs(0.01 * rng.standard_normal((k, S))))
        v = np.rint(np.exp(13.0 + rng.standard_normal((k, S))))
        last = c[-1]
        return [np.ascontiguousarray(x) for x in (c, h, lo, v)]

    def push(live, k, rows):
        eng.flush_l2()
        t = time.perf_counter()
        N.check(L.pqb_live_push(live._h, C.c_int64(k), *(r.ctypes.data_as(C.c_void_p) for r in rows), None, None, None, None, 1))
        return (time.perf_counter() - t) * 1e3, live.last_push_ms()

    res = {}
    for k in (1, 8, 64):
        times = {n: ([], []) for n in lives}
        for rep in range(3 + a.reps):
            rows = bars(k)                                 # the same bars into both, alternating which goes first
            order = list(lives) if rep % 2 == 0 else list(lives)[::-1]
            for n in order:
                e2e, dev = push(lives[n], k, rows)
                if rep >= 3:
                    times[n][0].append(dev)
                    times[n][1].append(e2e)
        r = {}
        for n, (dev, e2e) in times.items():
            r[n] = {"device_ms": float(np.median(dev)), "device_ms_min": float(np.min(dev)),
                    "e2e_ms": float(np.median(e2e)), "e2e_ms_min": float(np.min(e2e))}
        r["screen_extra_device_ms"] = r["screen"]["device_ms"] - r["plain"]["device_ms"]
        r["screen_extra_e2e_ms"] = r["screen"]["e2e_ms"] - r["plain"]["e2e_ms"]
        res["push_%d" % k] = r
    state = {n: lv.state_bytes for n, lv in lives.items()}
    bars_total = lives["screen"].bars
    for lv in lives.values():
        lv.close()

    # the whole-panel alternative: recompute the suite over T + 1 bars, then signals, MA cross and info
    full = pq.Panel(S, T + 1, outputs_mask=(1 << N.N_SUITE_OUTPUTS) - 1, host_staging=False)
    full.fill_synthetic(seed=0xC0FFEE, sigma=0.02)
    iters = 10
    tot, _, _ = full.time_device(params, warmup=3, iters=iters)
    sig_ms = C.c_float()
    N.check(L.pqb_signals_time(full._h, 30.0, 70.0, 3, iters, C.byref(sig_ms)))
    ma, info = [], []
    out_info = np.empty((len(N.INFO_NAMES), S))
    ok_info = np.empty((len(N.INFO_NAMES), S), dtype=np.uint8)
    for i in range(3 + iters):
        eng.flush_l2()
        t = time.perf_counter()
        N.check(L.pqb_ma_cross_run(full._h, 0, 10, 20))
        if i >= 3:
            ma.append((time.perf_counter() - t) * 1e3)
        eng.flush_l2()
        t = time.perf_counter()
        N.check(L.pqb_panel_info(full._h, out_info.ctypes.data, ok_info.ctypes.data))
        if i >= 3:
            info.append((time.perf_counter() - t) * 1e3)
    full.close()
    whole = {"suite_device_ms": tot / iters, "signals_device_ms": sig_ms.value / iters,
             "ma_cross_sma_10_20_ms": float(np.median(ma)), "info_ms": float(np.median(info))}
    whole["total_ms"] = sum(whole.values())
    name, power = card()
    out = {"metric": "live_screen_push", "symbols": S, "history_bars": T, "bars_after_pushes": bars_total,
           "screen": "macd / kdj / rsi cross, sma(10, 20) cross, info", "state_bytes_plain": state["plain"],
           "state_bytes_screen": state["screen"], "screen_extra_state_bytes": state["screen"] - state["plain"],
           "prime_ms_plain": prime_ms["plain"], "prime_ms_screen": prime_ms["screen"],
           "screen_extra_prime_ms": prime_ms["screen"] - prime_ms["plain"], **res,
           "whole_panel_%d_bars" % (T + 1): whole,
           "notes": "ma_cross / info of the whole panel: host clock around the synchronous call (kernel + launch; info "
                    "also copies its 13 rows to the host)",
           "gpu": name, "power_limit": power, "l2": "flushed before every timed push and call (pqb_flush_l2)", "reps": a.reps}
    line = json.dumps(out)
    print(line)
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
