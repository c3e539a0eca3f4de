"""Live panels at the benchmark shape: prime a 50,000 x 5,040 synthetic history once, then push k new random-walk bars
per symbol (k = 1, 8, 64) with a cold L2 before every timed push -- live bars arrive seconds apart -- and compare with one
device recompute of a 5,041-bar panel measured in the same run.  Prints one JSON line.

    python scripts/bench_live.py [--symbols 50000] [--bars 5040] [--reps 20] [--out file.json]

device_ms: CUDA events of pqb_live_push (pack of the new rows .. unpack of the result rows, no PCIe);
e2e_ms: host clock around pqb_live_push (host validation, H2D, kernels, D2H into pinned result rows).
bytes of a push = 2 x state_bytes (the state is read and written back) + the pushed rows in + the result rows out."""
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
    eng = pq.get_engine(0)
    params = N.default_params()
    L = N.lib()

    hist = pq.Panel(S, T, outputs_mask=0, host_staging=False)
    hist.fill_synthetic(seed=0xC0FFEE, sigma=0.02)
    t0 = time.perf_counter()
    live = pq.LivePanel(hist, params, None, 64)     # (create ends with a device synchronise)
    prime_ms = (time.perf_counter() - t0) * 1e3
    hist.close()
    state_bytes = live.state_bytes

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

    def push(k, rows):
        N.check(L.pqb_live_push(live._h, C.c_int64(k), *(r.ctypes.data_as(C.c_void_p) for r in rows), None, None, None, None, 1))

    n_out, n_in = len(live.outputs), 4
    res = {}
    for k in (1, 8, 64):
        for _ in range(3):
            push(k, bars(k))
        dev, e2e = [], []
        for _ in range(a.reps):
            rows = bars(k)
            eng.flush_l2()
            t = time.perf_counter()
            push(k, rows)
            e2e.append((time.perf_counter() - t) * 1e3)
            dev.append(live.last_push_ms())
        moved = 2 * state_bytes + k * S * 8 * (n_in + n_out) + k * ((S + 7) // 8) * n_out
        dm = float(np.median(dev))
        res["push_%d" % k] = {"device_ms": dm, "device_ms_min": float(np.min(dev)), "e2e_ms": float(np.median(e2e)),
                              "e2e_ms_min": float(np.min(e2e)), "bytes": moved, "achieved_GBps": moved / dm / 1e6}
    bars_total = live.bars
    live.close()

    full = pq.Panel(S, T + 1, outputs_mask=(1 << N.N_SUITE_OUTPUTS) - 1, host_staging=False)
    full.fill_synthetic(seed=0xC0FFEE, sigma=0.02)
    iters = 10
    tot, fused, nl = full.time_device(params, warmup=3, iters=iters)
    full.close()
    recompute_ms = tot / iters
    name, power = card()
    out = {"metric": "live_push", "symbols": S, "history_bars": T, "bars_after_pushes": bars_total, "outputs": n_out,
           "state_bytes": state_bytes, "prime_ms": prime_ms, **res,
           "recompute_%d_bars_device_ms" % (T + 1): recompute_ms,
           "push_1_over_recompute": res["push_1"]["device_ms"] / recompute_ms,
           "gpu": name, "power_limit": power, "l2": "flushed before every timed push (pqb_flush_l2)", "reps": a.reps}
    line = json.dumps(out)
    print(line)
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
