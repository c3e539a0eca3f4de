"""Live window panels at BASELINE config 5 (10,000 x 5,040; KDJ 5 / 9 / 14 / 60 / 250, WILLR / MIDPRICE / Donchian 5 / 20 /
55 / 250, ATR 14): prime a live window panel from a synthetic history once, then push k new random-walk bars per symbol
(k = 1, 8, 64) with a cold L2 before every timed push, and compare with a recompute of the 5,041-bar window panel, device
only (pqb_windows_time) and end to end (upload of the three input planes, run, download of the 32 output planes), all in
the same run.  Two histories: a clean one, and one with 1 % of the symbols halted 3 bars (every field), whose pushes carry
1 % of the symbols null in every bar.  Prints one JSON line.

    python scripts/bench_windows_live.py [--symbols 10000] [--bars 5040] [--reps 20] [--out file.json]

device_ms: CUDA events of pqb_windows_live_push (pack of the new rows .. unpack of the result rows and the move of the
high / low tail, no PCIe); e2e_ms: host clock around pqb_windows_live_push (null rules on the host, H2D, kernels, D2H into
pinned result rows)."""
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
from polars_quant_b200.windows import WindowPanel   # noqa: E402

KDJ, EXT, ATR = (5, 9, 14, 60, 250), (5, 20, 55, 250), 14


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = (x.strip() for x in q.split(","))
        return name, power
    except Exception as ex:                          # (reported, not guessed)
        return "unknown (%s)" % ex, "unknown"


def history(S, T, halted, rng):
    wp = WindowPanel(S, T, kdj=KDJ, ext=EXT, atr=ATR, host_staging=True)
    wp.panel.fill_synthetic(seed=0xC0FFEE, sigma=0.02, to_host=True)
    if halted:                                       # 1 % of the symbols halted (every field null) for 3 bars
        for s in rng.choice(S, S // 100, replace=False):
            ok = np.ones(T, dtype=bool)
            a = int(rng.integers(100, T - 3))
            ok[a:a + 3] = False
            bits = np.packbits(ok, bitorder="little")
            for f in range(3):
                wp.panel.set_column(int(s), f, wp.panel.host_field(f)[s, :T].copy(), validity=bits)
    wp.panel.upload()
    return wp


def pushes(live, S, reps, nulls, rng):
    eng, L = pq.get_engine(0), N.lib()
    last = np.full(S, 100.0)

    def bars(k):
        nonlocal last
        c = last * np.exp(np.cumsum(0.02 * rng.standard_normal((k, S)), axis=0))
        o = np.vstack([last[None, :], c[:-1]])
        h = np.maximum(o, c) * (1.0 + np.abs(0.01 * rng.standard_normal((k, S))))
        lo = np.minimum(o, c) * (1.0 - np.abs(0.01 * rng.standard_normal((k, S))))
        last = c[-1]
        vb = None
        if nulls:
            ok = np.ones((k, S), dtype=bool)
            for t in range(k):
                ok[t, rng.choice(S, S // 100, replace=False)] = False
            vb = np.ascontiguousarray(np.packbits(ok, axis=1, bitorder="little"))
        return [np.ascontiguousarray(x) for x in (c, h, lo)], vb

    def push(k):
        rows, vb = bars(k)
        ptr = lambda x: None if x is None else x.ctypes.data_as(C.c_void_p)
        eng.flush_l2()
        t = time.perf_counter()
        N.check(L.pqb_windows_live_push(live._h, C.c_int64(k), *(ptr(r) for r in rows), *([ptr(vb)] * 3), 1))
        return (time.perf_counter() - t) * 1e3

    res = {}
    for k in (1, 8, 64):
        for _ in range(3):
            push(k)
        dev, e2e = [], []
        for _ in range(reps):
            e2e.append(push(k))
            dev.append(live.last_push_ms())
        res["push_%d" % k] = {"device_ms": float(np.median(dev)), "device_ms_min": float(np.min(dev)),
                              "e2e_ms": float(np.median(e2e)), "e2e_ms_min": float(np.min(e2e))}
    return res


def recompute(S, T, halted, rng):
    """the (T + 1)-bar window panel: device time of one run, and upload + run + download end to end"""
    wp = history(S, T + 1, halted, rng)
    dev_total, launches = wp.time_device(warmup=2, iters=10)
    e2e = []
    for _ in range(4):
        t = time.perf_counter()
        wp.panel.upload()
        wp.run()
        wp.panel.download()
        wp.panel.sync()
        e2e.append((time.perf_counter() - t) * 1e3)
    wp.close()
    return {"device_ms": dev_total, "launches": launches, "e2e_ms": float(np.median(e2e[1:])), "e2e_ms_min": float(np.min(e2e[1:]))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--symbols", type=int, default=10000)
    ap.add_argument("--bars", type=int, default=5040)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    S, T = a.symbols, a.bars
    rng = np.random.default_rng(7)
    out = {"metric": "windows_live_push", "symbols": S, "history_bars": T, "kdj": KDJ, "ext": EXT, "atr": ATR,
           "lines": 3 * len(KDJ) + 4 * len(EXT) + 1}
    for tag, halted in (("clean", False), ("halted", True)):
        wp = history(S, T, halted, rng)
        t0 = time.perf_counter()
        live = wp.live(64)                           # (create ends with a device synchronise)
        r = {"prime_ms": (time.perf_counter() - t0) * 1e3, "state_bytes": live.state_bytes}
        wp.close()
        r.update(pushes(live, S, a.reps, halted, rng))
        live.close()
        r["recompute_%d_bars" % (T + 1)] = recompute(S, T, halted, rng)
        r["push_1_device_over_recompute_device"] = r["push_1"]["device_ms"] / r["recompute_%d_bars" % (T + 1)]["device_ms"]
        r["push_1_e2e_over_recompute_e2e"] = r["push_1"]["e2e_ms"] / r["recompute_%d_bars" % (T + 1)]["e2e_ms"]
        out[tag] = r
    out["halts"] = "halted: 1 % of the symbols 3 bars (every field) in the history; 1 % of the symbols null in every pushed bar"
    name, power = card()
    out.update({"gpu": name, "power_limit": power, "l2": "flushed before every timed push (pqb_flush_l2)", "reps": a.reps})
    line = json.dumps(out)
    print(line)
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
