"""Live panels at the benchmark shape: prime a 50,000 x 5,040 synthetic history once, then push k new random-walk bars
per symbol (k = 1, 8, 64) with a cold L2 before every timed push -- live bars arrive seconds apart -- and compare with one
device recompute of a 5,041-bar panel measured in the same run.  Prints one JSON line.

    python scripts/bench_live.py [--symbols 50000] [--bars 5040] [--reps 20] [--out file.json] [--nulls]

--nulls: the null-aware live panel (LivePanel(..., nulls=True)) on a history in which 1 % of the symbols have a 3-bar halt
(all fields), with 1 % of the symbols null in every pushed bar, beside the strict live panel on the clean history and a
device recompute of both 5,041-bar panels -- all in the same run.

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
    ap.add_argument("--nulls", action="store_true")
    a = ap.parse_args()
    if a.nulls:
        return main_nulls(a)
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


def halted_panel(S, n, rng, outputs_mask):
    """synthetic S x n panel, 1 % of the symbols halted (every field null) for 3 bars"""
    p = pq.Panel(S, n, outputs_mask=outputs_mask, host_staging=True)
    p.fill_synthetic(seed=0xC0FFEE, sigma=0.02, to_host=True)
    for s in rng.choice(S, S // 100, replace=False):
        ok = np.ones(n, dtype=bool)
        a = int(rng.integers(100, n - 3))
        ok[a:a + 3] = False
        bits = np.packbits(ok, bitorder="little")
        for f in range(4):
            p.set_column(int(s), f, p.host_field(f)[s, :n].copy(), validity=bits)
    p.upload()
    return p


def push_times(live, S, reps, valid_fn):
    """median / min device and end-to-end ms of pushes of k = 1, 8, 64 random-walk bars, cold L2 before each"""
    eng, L = pq.get_engine(0), N.lib()
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

    def push(k):
        rows, vb = bars(k), valid_fn(k)
        ptr = lambda x: None if x is None else x.ctypes.data_as(C.c_void_p)
        t = time.perf_counter()
        N.check(L.pqb_live_push(live._h, C.c_int64(k), *(ptr(r) for r in rows), *([ptr(vb)] * 4), 1))
        return (time.perf_counter() - t) * 1e3

    res = {}
    for k in (1, 8, 64):
        for _ in range(3):
            push(k)
        dev, e2e = [], []
        for _ in range(reps):
            eng.flush_l2()
            e2e.append(push(k))
            dev.append(live.last_push_ms())
        res["push_%d" % k] = {"device_ms": float(np.median(dev)), "device_ms_min": float(np.min(dev)),
                              "e2e_ms": float(np.median(e2e)), "e2e_ms_min": float(np.min(e2e))}
    return res


def main_nulls(a):
    S, T = a.symbols, a.bars
    params = N.default_params()
    rng = np.random.default_rng(7)
    out = {"metric": "live_push_nulls", "symbols": S, "history_bars": T,
           "halts": "1 % of the symbols: 3 bars, every field; pushes: 1 % of the symbols null in every bar"}
    # strict live panel, clean history
    hist = pq.Panel(S, T, outputs_mask=0, host_staging=False)
    hist.fill_synthetic(seed=0xC0FFEE, sigma=0.02)
    t0 = time.perf_counter()
    live = pq.LivePanel(hist, params, None, 64)
    strict = {"prime_ms": (time.perf_counter() - t0) * 1e3}
    hist.close()
    strict["state_bytes"] = live.state_bytes
    strict.update(push_times(live, S, a.reps, lambda k: None))
    live.close()
    out["strict_clean_history"] = strict
    # null-aware live panel, halted history, pushes with nulls
    hist = halted_panel(S, T, rng, 0)
    t0 = time.perf_counter()
    live = pq.LivePanel(hist, params, None, 64, nulls=True)
    nl = {"prime_ms": (time.perf_counter() - t0) * 1e3}
    hist.close()
    nl["state_bytes"] = live.state_bytes
    vb = (S + 7) // 8

    def valid(k):
        ok = np.ones((k, S), dtype=bool)
        for t in range(k):
            ok[t, rng.choice(S, S // 100, replace=False)] = False
        return np.ascontiguousarray(np.packbits(ok, axis=1, bitorder="little")[:, :vb])

    nl.update(push_times(live, S, a.reps, valid))
    nl["bars_after_pushes"] = live.bars
    live.close()
    out["nulls"] = nl
    # device recomputes of the 5,041-bar panels
    iters = 10
    full = pq.Panel(S, T + 1, outputs_mask=(1 << N.N_SUITE_OUTPUTS) - 1, host_staging=False)
    full.fill_synthetic(seed=0xC0FFEE, sigma=0.02)
    out["recompute_clean_%d_bars_device_ms" % (T + 1)] = full.time_device(params, warmup=3, iters=iters)[0] / iters
    full.close()
    full = halted_panel(S, T + 1, np.random.default_rng(7), (1 << N.N_SUITE_OUTPUTS) - 1)
    out["recompute_halted_%d_bars_device_ms" % (T + 1)] = full.time_device(params, warmup=3, iters=iters)[0] / iters
    full.close()
    name, power = card()
    out.update({"gpu": name, "power_limit": power, "l2": "flushed before every timed push (pqb_flush_l2)", "reps": a.reps})
    line = json.dumps(out)
    print(line)
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
