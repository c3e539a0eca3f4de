#!/usr/bin/env python
"""Optional indicator groups on a halted panel: 50,000 symbols x 5,040 bars, device-resident, clean and with 1 % / 5 % / 20 % of
the symbols (spread evenly) halted for 3 bars in close, as in bench_halted_symbols.py.  Kernel time per pass of
(a) the suite plus every optional group, (b) the DM family alone, (c) CCI alone -- and the suite alone beside them.  Prints one JSON line per case, the first one
with the card's name and power limit."""
import json, os, subprocess, sys
from pathlib import Path
import numpy as np
ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
import polars_quant_b200 as pq
from polars_quant_b200 import _native as N

S, NB = int(os.environ.get("PQB_BENCH_SYMBOLS", 50000)), 5040
ITERS = int(os.environ.get("PQB_BENCH_ITERS", 5))
card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                      capture_output=True, text=True).stdout.strip()
print(json.dumps({"card": card, "symbols": S, "bars": NB, "iters": ITERS}), flush=True)
CASES = {"suite alone": N.IND_ALL, "suite + every optional group": N.IND_ALL | sum(N.IND_EXTRA.values()),
         "dm alone": N.IND_EXTRA["dm"], "cci alone": N.IND_EXTRA["cci"]}
outputs = (1 << N.N_OUTPUTS) - 1 - (1 << N.OUTPUT_NAMES.index("fastk"))
p = pq.Panel(S, NB, engine=pq.get_engine(0), outputs_mask=outputs)
p.fill_synthetic(seed=5, to_host=True)
base = {}
ok = np.ones(NB, dtype=bool); ok[2000:2003] = False
bits = np.packbits(ok, bitorder="little")
for frac in (0.0, 0.01, 0.05, 0.2):
    halted = np.arange(0, S, round(1 / frac)) if frac else np.arange(0)     # (each set holds the previous one)
    for s in halted:
        p.set_column(int(s), "close", np.ascontiguousarray(p.host_field("close")[int(s)]), validity=bits)
    p.upload()
    for name, ind in CASES.items():
        tot, fused, nl = p.time_device(N.default_params(indicators=ind), warmup=2, iters=ITERS)
        ms = tot / ITERS
        if frac == 0.0:
            base[name] = ms
        print(json.dumps({"case": name, "halted_symbols": len(halted), "halted_pct": 100 * frac, "ms_per_pass": round(ms, 3),
                          "vs_clean": round(ms / base[name], 3), "launches": nl}), flush=True)
p.close()
