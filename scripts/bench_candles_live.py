"""Live candle panels at the candle bench shape (20,000 x 5,040 busy synthetic candles, all 61 patterns + the 4 price
transforms + BOP): prime a live candle panel from the device-resident history once, then push k new bars per symbol
(k = 1, 8, 64) with a cold L2 before every timed push, and compare with a recompute of the panel, device only
(pqb_candles_time) and end to end (pqb_candles_run_host: upload, kernel, download of every output plane), all in the same
run.  Prints one JSON line.

    python scripts/bench_candles_live.py [--symbols 20000] [--bars 5040] [--reps 20] [--out file.json]

device_ms: CUDA events of pqb_candles_live_push (H2D of the pushed rows .. end of the walk; the result rows' D2H is not
included); e2e_ms: host clock around pqb_candles_live_push (null checks and staging on the host, H2D, kernel, D2H into
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
from polars_quant_b200 import candles               # noqa: E402

IN_BYTES = 4 * 8                                    # open / high / low / close
OUT_BYTES = 61 * 4 + 5 * 8                          # result rows per symbol and bar (+ 5 validity bits)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = (x.strip() for x in q.split(","))
        return name, power
    except Exception as ex:                          # (reported, not guessed)
        return "unknown (%s)" % ex, "unknown"


def pushes(live, S, reps, eng):
    """k-bar pushes of bar-major rows cut from a 128-bar busy synthetic panel (the kernel's work does not depend on the
    values: every enabled pattern is evaluated at every bar)"""
    L = N.lib()
    pool = candles.CandlePanel(S, 128, engine=eng, patterns_mask=0, prices_mask=0)
    pool.fill_synthetic(seed=11, to_host=True)
    rows = [np.ascontiguousarray(pool.host_field(f).T) for f in range(4)]      # [128][S]
    pool.close()
    state = {"at": 0}

    def push(k):
        a = state["at"] % (128 - k + 1)
        state["at"] += 7
        p = [r[a:a + k].ctypes.data_as(C.c_void_p) for r in rows]
        eng.flush_l2()
        t = time.perf_counter()
        N.check(L.pqb_candles_live_push(live._h, C.c_int64(k), *p, None, None, None, None, 1))
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
                              "e2e_ms": float(np.median(e2e)), "e2e_ms_min": float(np.min(e2e)),
                              "h2d_bytes": IN_BYTES * S * k, "d2h_bytes": OUT_BYTES * S * k + 5 * ((S + 7) // 8) * k}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--symbols", type=int, default=20000)
    ap.add_argument("--bars", type=int, default=5040)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    S, T = a.symbols, a.bars
    eng = pq.get_engine(0)
    out = {"metric": "candles_live_push", "symbols": S, "history_bars": T, "patterns": 61, "prices": 5,
           "data": "busy synthetic candles (pqb_candles_fill_synthetic)"}
    p = candles.CandlePanel(S, T, engine=eng, host_staging=True)
    p.fill_synthetic(seed=3, to_host=True)
    iters = 10
    rec = {"device_ms": p.time_device(warmup=3, iters=iters) / iters}
    p.run_host()
    e2e = []
    for _ in range(3):
        t = time.perf_counter()
        p.run_host()
        e2e.append((time.perf_counter() - t) * 1e3)
    rec.update({"e2e_ms": float(np.median(e2e)), "e2e_ms_min": float(np.min(e2e)),
                "h2d_bytes": IN_BYTES * S * T, "d2h_bytes": OUT_BYTES * S * T})
    out["recompute_%d_bars" % T] = rec
    t0 = time.perf_counter()
    live = p.live(max_push_bars=64)                  # (create ends with a device synchronise)
    out["prime_ms"] = (time.perf_counter() - t0) * 1e3
    p.close()
    out.update(pushes(live, S, a.reps, eng))
    live.close()
    out["push_1_device_over_recompute_device"] = out["push_1"]["device_ms"] / rec["device_ms"]
    out["push_1_e2e_over_recompute_e2e"] = out["push_1"]["e2e_ms"] / rec["e2e_ms"]
    name, power = card()
    out.update({"gpu": name, "power_limit": power, "l2": "flushed before every timed push (pqb_flush_l2)", "reps": a.reps})
    line = json.dumps(out)
    print(line)
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
