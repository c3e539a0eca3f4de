#!/usr/bin/env python
"""Config 5 (10,000 x 5,040: KDJ 5 / 9 / 14 / 60 / 250, WILLR / MIDPRICE / Donchian 5 / 20 / 55 / 250, ATR 14) on panels with
halted symbols, device-resident: kernel time per pass (CUDA events over pqb_windows_time), clean and with 1 %, 5 % and 20 % of
the symbols (spread evenly) halted for 3 bars in close, high and low, and how many of the 313 symbol blocks each share flags.

--baseline-lib PATH also times the clean panel with another build of the library (the parent commit's, say): the two builds
alternate, ROUNDS times each, every timing in a process of its own.  The card's name and power limit are read in the same run.
Writes one JSON document to --out (default profiles/r10_bench_windows_nulls.json) and prints it."""
import argparse, json, os, subprocess, sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

S, NB = 10_000, 5_040
KDJ, EXT, ATR = (5, 9, 14, 60, 250), (5, 20, 55, 250), 14


def clean_ms(warmup, iters):
    from polars_quant_b200.windows import WindowPanel
    wp = WindowPanel(S, NB, kdj=KDJ, ext=EXT, atr=ATR, host_staging=False)
    wp.fill_synthetic(seed=55, sigma=0.02)
    ms, nl = wp.time_device(warmup=warmup, iters=iters)
    wp.close()
    return ms, nl


def halted_cases(warmup, iters):
    from polars_quant_b200.windows import WindowPanel
    wp = WindowPanel(S, NB, kdj=KDJ, ext=EXT, atr=ATR)
    wp.fill_synthetic(seed=55, sigma=0.02, to_host=True)
    ok = np.ones(NB, dtype=bool)
    ok[2000:2003] = False
    bits = np.packbits(ok, bitorder="little")
    n_blocks = (S + 31) // 32
    out = []
    for frac in (0.01, 0.05, 0.2):
        halted = np.arange(0, S, round(1 / frac))                 # (each set holds the previous one)
        for s in halted:
            for f in ("close", "high", "low"):
                wp.panel.set_column(int(s), f, np.ascontiguousarray(wp.panel.host_field(f)[int(s)]), validity=bits)
        wp.panel.upload()
        ms, nl = wp.time_device(warmup=warmup, iters=iters)
        out.append({"halted_pct": 100 * frac, "halted_symbols": int(len(halted)),
                    "flagged_blocks": int(len(set(int(s) // 32 for s in halted))), "blocks": n_blocks,
                    "ms_per_pass": round(ms, 4), "launches": nl})
    wp.close()
    return out


def child(which, lib, warmup, iters):
    env = dict(os.environ)
    if lib:
        env["PQB_LIB"] = str(lib)
    else:
        env.pop("PQB_LIB", None)
    r = subprocess.run([sys.executable, __file__, "--child", which, "--warmup", str(warmup), "--iters", str(iters)],
                       env=env, capture_output=True, text=True, check=True)
    return json.loads(r.stdout.strip().splitlines()[-1])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--baseline-lib", default=None, help="another libpqb200.so to time the clean panel with, alternating")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r10_bench_windows_nulls.json"))
    ap.add_argument("--child", choices=("clean", "halted"), help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.child == "clean":
        ms, nl = clean_ms(a.warmup, a.iters)
        print(json.dumps({"ms_per_pass": ms, "launches": nl}))
        return
    if a.child == "halted":
        print(json.dumps(halted_cases(a.warmup, a.iters)))
        return
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                          capture_output=True, text=True).stdout.strip()
    doc = {"card": card, "symbols": S, "bars": NB, "kdj": KDJ, "ext": EXT, "atr": ATR, "warmup": a.warmup, "iters": a.iters}
    clean = {"this build": []}
    if a.baseline_lib:
        clean["baseline build"] = []
    for _ in range(a.rounds):
        for name in clean:
            r = child("clean", a.baseline_lib if name == "baseline build" else None, a.warmup, a.iters)
            clean[name].append(round(r["ms_per_pass"], 4))
            doc.setdefault("clean_launches", {})[name] = r["launches"]
    doc["clean_ms_per_pass"] = clean
    doc["clean_median_ms"] = {k: float(np.median(v)) for k, v in clean.items()}
    doc["halted"] = child("halted", None, a.warmup, a.iters)
    med = doc["clean_median_ms"]["this build"]
    for h in doc["halted"]:
        h["vs_clean"] = round(h["ms_per_pass"] / med, 3)
    text = json.dumps(doc, indent=1)
    Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    Path(a.out).write_text(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
