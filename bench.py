#!/usr/bin/env python
"""bench.py -- fused indicator suite throughput (symbol.bars/s) on B200, one JSON line.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c4|c2|c3|c5] [--dump-outputs DIR]

A "step" is one pass of the fused 15-indicator / 21-output suite over one synthetic random-walk
OHLCV panel already resident in HBM.  N > 1 is launched by torchrun, one process per GPU; symbols
are independent, so the workload's 50,000 symbols are SHARDED over the ranks in contiguous ranges of
whole 32-symbol blocks (strong scaling -- BASELINE config 4; `--scaling weak` runs the full shape on
every rank), with no collective on the data path; torch.distributed (NCCL) is used only for the
barrier and the max-over-ranks of the timed durations.

Keys beyond the base contract:
  roofline      dominant kernel (suite_fused_kernel) vs the measured HBM copy peak
  cpu_baseline  the C oracle (a port of the reference's Rust loops) on this box's host cores
  e2e           same metric through the public column API: caller-owned column buffers in (pageable host memory),
                Arrow result columns out, every host copy and both PCIe directions inside the timed region
`--impl reference` times the reference's own CPU path -- the C oracle port, since the Rust crate
cannot be built in this image -- on all host cores, same config/metric/unit.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

WORKLOADS = {
    # name: (symbols, bars, description)
    "c4": (50_000, 5_040, "BASELINE config 4 / north_star target: 50,000 symbols x 5,040 bars f64 OHLCV, full 15-indicator suite"),
    "c2": (5_000, 2_520, "BASELINE config 2: 5,000 symbols x 2,520 bars f64 OHLCV, full 15-indicator suite"),
}
N_IN, N_OUT = 4, 21
ALGO_BYTES_PER_SYMBOL_BAR = 8 * (N_IN + N_OUT)          # 200 B (SURVEY.md 8d); validity bits (+2.6 B) not counted
METRIC = "symbol_bars_per_sec_fused_indicator_suite"
UNIT = "symbol*bars/s"
DUMP_BYTES = 64_000_000                                  # --dump-outputs: all files together stay below this
DUMP_SEED = 0x5EED


def measured_peak():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region: NVML in-process every ~5 ms
    (nvidia_ml_py), falling back to polling nvidia-smi."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.sm, self.mx, self.reasons = [], [], set()
        self._stop = threading.Event()
        self._t = None
        self._nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self._h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
            self._nvml = pynvml
        except Exception:
            self._nvml = None

    def _run_nvml(self):
        nv = self._nvml
        names = {"hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4)}
        get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
            getattr(nv, "nvmlDeviceGetCurrentClocksThrottleReasons")
        try:
            mx = float(nv.nvmlDeviceGetMaxClockInfo(self._h, nv.NVML_CLOCK_SM))
        except Exception:
            mx = None
        while not self._stop.is_set():
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM)))
                if mx:
                    self.mx.append(mx)
                r = int(get_reasons(self._h))
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            self._stop.wait(0.005)

    def _run_smi(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                for line in out.strip().splitlines():
                    r = [c.strip() for c in line.split(",")]
                    self.sm.append(float(r[1])); self.mx.append(float(r[2]))
                    for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                        if v.lower().startswith("active"):
                            self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(0.05)

    def __enter__(self):
        self._t = threading.Thread(target=self._run_nvml if self._nvml else self._run_smi, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        if not self.sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(self.sm)), "sm_max_mhz": float(max(self.mx)) if self.mx else None,
                "reasons": sorted(self.reasons), "samples": len(self.sm),
                "source": "nvml" if self._nvml else "nvidia-smi"}


def cpu_suite_rate(c, h, l, v, threads: int, budget_s: float):
    """Times the C oracle (reference port) over [symbols, bars] host arrays; repeats to ~budget."""
    from oracle import pqo
    S, N = c.shape
    t0 = time.perf_counter()
    _, _, used = pqo.suite_panel(c, h, l, v, threads=threads)
    dt = time.perf_counter() - t0
    reps, total = 1, dt
    while total < budget_s and reps < 50:
        t0 = time.perf_counter()
        pqo.suite_panel(c, h, l, v, threads=threads)
        total += time.perf_counter() - t0
        reps += 1
    return S * N * reps / total, used, reps


def synth_host_sample(n_symbols, n_bars, seed=0xC0FFEE):
    import synth
    d = synth.ohlcv(n_symbols, n_bars, seed=seed)
    return d["close"], d["high"], d["low"], d["volume"]


def dump_outputs(panel, out_dir):
    """Writes the 21 result columns of the panel's last suite run as a caller receives them, values and validity:
    out_dir/<output>.npy, float64 [symbols, bars], 0.0 where the value is null, and out_dir/<output>_valid.npy, float32,
    1.0 where the validity bit is set and 0.0 where it is clear.  Covers a fixed seeded sample of the panel's symbols
    small enough to keep the files within DUMP_BYTES.  Read from the tiled device planes."""
    import devread
    from polars_quant_b200 import _native as NV
    S, N = panel.n_symbols, panel.n_bars
    k = min(S, (DUMP_BYTES - 2 * 4096 * N_OUT) // (N_OUT * N * (8 + 4)))
    if k < 1:
        raise SystemExit("--dump-outputs: one symbol's %d outputs over %d bars exceed %d bytes" % (N_OUT, N, DUMP_BYTES))
    syms = np.sort(np.random.default_rng(DUMP_SEED).choice(S, size=k, replace=False))
    _, bars_padded = panel.tiled_shape()
    os.makedirs(out_dir, exist_ok=True)
    for j, name in enumerate(NV.OUTPUT_NAMES[:N_OUT]):
        vals_ptr = NV.lib().pqb_panel_device_output(panel._h, j)
        bits_ptr = NV.lib().pqb_panel_device_validity(panel._h, j)
        out = np.empty((k, N), dtype=np.float64)
        valid = np.empty((k, N), dtype=bool)
        for b in np.unique(syms // 32):
            rows = np.flatnonzero(syms // 32 == b)
            vals = devread.read_block(vals_ptr, int(b), bars_padded, N)
            ok = devread.read_validity_rows(bits_ptr, int(b) * 32, min(32, S - int(b) * 32), panel.validity_pitch, N)
            lanes = syms[rows] % 32
            valid[rows] = ok[lanes]
            out[rows] = np.where(ok[lanes], vals[lanes], 0.0)
        np.save(os.path.join(out_dir, name + ".npy"), out)
        np.save(os.path.join(out_dir, name + "_valid.npy"), valid.astype(np.float32))
    sys.stderr.write("[bench] wrote %d outputs of symbols %s (of %d) x %d bars to %s\n"
                     % (N_OUT, syms.tolist(), S, N, out_dir))


def run_reference(args, shape, rank, world):
    """--impl reference: the reference's CPU path (oracle port; oracle/_ref does not exist because
    the Rust reference cannot be compiled here) on all host cores.  Rank 0 only."""
    if rank != 0:
        return
    S, N, desc = shape
    cores = os.cpu_count() or 1
    # bounded sample of the workload: enough symbols for ~1-2 s per step on this box
    sample_symbols = min(S, max(64, 16 * cores))
    c, h, l, v = synth_host_sample(sample_symbols, N)
    from oracle import pqo
    for _ in range(max(args.warmup, 1)):
        pqo.suite_panel(c, h, l, v, threads=cores)
    t0 = time.perf_counter()
    used = cores
    for _ in range(args.steps):
        _, _, used = pqo.suite_panel(c, h, l, v, threads=cores)
    dt = time.perf_counter() - t0
    value = sample_symbols * N * args.steps / dt
    sample = f"{sample_symbols} of {S} symbols x {N} bars per step, numpy random-walk OHLCV, {used} threads"
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": getattr(args, "scaling", "strong"), "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": desc, "symbols": S, "bars": N, "sample": sample},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": used, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def traffic_record(S, N):
    """ncu DRAM bytes of the dominant kernel for this shape, with the commit it was captured at (profiles/traffic.json,
    written by scripts/ncu_traffic.sh from an `ncu --set full` capture; never measured under the timer)."""
    tp = ROOT / "profiles" / "traffic.json"
    if not tp.exists():
        return None, None
    try:
        tj = json.loads(tp.read_text())
        for rec in (tj if isinstance(tj, list) else [tj]):
            if rec.get("symbols") == S and rec.get("bars") == N:
                return rec.get("dram_bytes_per_launch"), {k: rec.get(k) for k in ("captured_at_commit", "kernel", "source") if rec.get(k)}
    except Exception:
        pass
    return None, None


def bench_c3(pq, NV, engine, peak, iters=5, warmup=2):
    """BASELINE config 3: 500 x 1,000,000, EMA(12, 26, 200, 5000) + MACD(12, 26, 9): 1 plane in, 7 out = 64 B per
    symbol-bar (SURVEY.md 8d)."""
    from polars_quant_b200 import longrows
    S, NB = 500, 1_000_000
    lp = longrows.LongPanel(S, NB, engine=engine, ema_periods=(12, 26, 200, 5000), macd=(12, 26, 9), host_staging=False)
    lp.fill_synthetic(seed=3, sigma=0.0005)
    ms, launches = lp.time_device(warmup=warmup, iters=iters)
    lp.close()
    g = 64 * S * NB / (ms * 1e-3) / 1e9
    return {"workload": "BASELINE config 3: 500 symbols x 1,000,000 minute bars, EMA(12,26,200,5000) + MACD(12,26,9) in one pass",
            "kernel": "lr_local_kernel + lr_carry_kernel + lr_final_kernel", "launches": launches, "kernel_ms": ms, "value": S * NB / (ms * 1e-3), "unit": UNIT,
            "algorithmic_bytes_per_symbol_bar": 64, "achieved_gbs": g, "frac": g / peak}


def bench_c5(pq, NV, engine, peak, iters=5, warmup=2):
    """BASELINE config 5: 10,000 x 5,040, KDJ(k) for k in 5/9/14/60/250 + WILLR / MIDPRICE / Donchian(p) for p in
    5/20/55/250 + ATR(14): 3 planes in, 28 out = 248 B per symbol-bar (SURVEY.md 8d)."""
    from polars_quant_b200 import windows
    S, NB = 10_000, 5_040
    wp = windows.WindowPanel(S, NB, engine=engine, kdj=(5, 9, 14, 60, 250), ext=(5, 20, 55, 250), atr=14, host_staging=False)
    wp.fill_synthetic(seed=55, sigma=0.02)
    ms, launches = wp.time_device(warmup=warmup, iters=iters)
    wp.close()
    g = 248 * S * NB / (ms * 1e-3) / 1e9
    return {"workload": "BASELINE config 5: 10,000 x 5,040, KDJ(5,9,14,60,250) + WILLR/MIDPRICE/Donchian(5,20,55,250) + ATR(14)",
            "kernel": "window_suite_kernel", "launches": launches, "kernel_ms": ms, "value": S * NB / (ms * 1e-3), "unit": UNIT,
            "algorithmic_bytes_per_symbol_bar": 248, "achieved_gbs": g, "frac": g / peak}


def run_config_3_or_5(args, rank):
    """`--workload c3|c5`: the long-row / many-window panels as a bench line of their own (device-resident, one GPU; under
    torchrun every rank but 0 exits).  Same timing rules: W >= 3 warm-up passes, K timed passes between CUDA events on the engine
    stream; inputs + outputs per pass (12.5 - 32 GB) dwarf the L2."""
    if rank != 0:
        return
    import polars_quant_b200 as pq
    from polars_quant_b200 import _native as NV
    engine = pq.get_engine(0)
    peak, peak_src = measured_peak()
    with ClockSampler(0) as clocks:
        rec = (bench_c3 if args.workload == "c3" else bench_c5)(pq, NV, engine, peak, iters=max(args.steps, 1), warmup=max(args.warmup, 3))
    S, NB = (500, 1_000_000) if args.workload == "c3" else (10_000, 5_040)
    line = {"metric": "symbol_bars_per_sec_" + ("ema_macd_long_rows" if args.workload == "c3" else "rolling_window_suite"),
            "value": rec["value"], "unit": UNIT, "n_gpus": 1, "steps": max(args.steps, 1), "warmup": max(args.warmup, 3),
            "ms_per_step": rec["kernel_ms"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic", "config": {"workload": rec["workload"], "symbols": S, "bars": NB,
                                            "l2": "inputs + outputs per pass are far larger than the 126 MB L2; no flush needed"},
            "roofline": {"bound": "hbm", "achieved": rec["achieved_gbs"], "peak": peak, "unit": "GB/s", "frac": rec["frac"],
                         "traffic": None, "kernel": rec["kernel"], "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": rec["algorithmic_bytes_per_symbol_bar"] * S * NB, "kernel_ms": rec["kernel_ms"]},
            "cpu_baseline": None, "e2e": None, "gpu_launches": rec["launches"] * max(args.steps, 1), "clocks": clocks.summary()}
    tr = ROOT / "profiles" / "traffic.json"
    try:
        for r in json.loads(tr.read_text()):
            if r.get("workload") == args.workload:
                line["roofline"]["traffic"] = r.get("dram_bytes_per_launch")
                line["roofline"]["traffic_source"] = {k: r.get(k) for k in ("captured_at_commit", "kernel")}
    except Exception:
        pass
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c4", choices=sorted(WORKLOADS) + ["c3", "c5"],
                    help="c4 (default) / c2: the fused suite; c3: EMA x 4 + MACD over 500 x 1,000,000 (LongPanel); c5: KDJ x 5 + WILLR / "
                         "MIDPRICE / Donchian x 4 + ATR over 10,000 x 5,040 (WindowPanel) -- kernel-only lines, one GPU")
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"],
                    help="strong (default): the workload's symbols are sharded over the GPUs (BASELINE config 4: '50,000 x 5,040 "
                         "symbol-sharded at 1/2/4/8'); weak: every GPU runs the whole workload shape")
    ap.add_argument("--symbols", type=int, default=0, help="override the workload's symbol count")
    ap.add_argument("--bars", type=int, default=0)
    ap.add_argument("--no-extra", action="store_true", help="skip the kernel-only lines of the other shapes (configs 2, 3, 5, candles)")
    ap.add_argument("--e2e-symbols", type=int, default=0, help="symbols per GPU pushed through the column API (0: the GPU's whole share)")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--threads", type=int, default=0, help="host threads of the column intake per GPU (0: cores / GPUs, at most 6)")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the fused suite's 21 outputs of the last step for a fixed seeded sample of "
                         "symbols as DIR/<output>.npy (float64, 0.0 where null) and DIR/<output>_valid.npy (float32, 1.0 where "
                         "valid), under 64 MB in all; rank 0's share under torchrun")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.workload not in WORKLOADS):
        ap.error("--dump-outputs writes the fused suite's outputs: --impl ours with --workload %s" % " or ".join(sorted(WORKLOADS)))
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.workload in ("c3", "c5"):
        if args.impl == "reference":
            if rank == 0:
                print(json.dumps({"impl": "reference", "unavailable": "the reference arm is timed on the headline workloads (c4 / c2) only"}), flush=True)
            return
        run_config_3_or_5(args, rank)
        return
    S_total, N, desc = WORKLOADS[args.workload]
    if args.symbols:
        S_total = args.symbols
    if args.bars:
        N = args.bars

    if args.impl == "reference":
        run_reference(args, (S_total, N, desc), rank, world)
        return

    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        # NCCL prints its version banner (NCCL_DEBUG=VERSION/INFO in some images) on stdout: keep stdout
        # to the one JSON line of the contract
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        # ... and some builds print it with a plain printf when the communicator is created: point fd 1 at stderr
        # until the first collective has run
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_stdout, 1)
            os.close(saved_stdout)

    import polars_quant_b200 as pq
    from polars_quant_b200 import _native as NV
    from polars_quant_b200.shard import symbol_range

    def barrier():
        if dist is not None:
            dist.barrier()

    def max_over_ranks(*vals):
        if dist is None:
            return vals
        import torch
        t = torch.tensor(list(vals), dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return tuple(float(x) for x in t)

    # this GPU's share of the panel: contiguous whole 32-symbol blocks (SURVEY.md 8e), or the whole shape (weak)
    if args.scaling == "strong":
        lo, hi = symbol_range(S_total, world, rank)
        S = hi - lo
        units = S_total * N
    else:
        lo, S = 0, S_total
        units = S_total * N * world

    engine = pq.get_engine(local_rank)
    params = NV.default_params()
    panel = pq.Panel(S, N, engine=engine, host_staging=False)
    panel.fill_synthetic(seed=0xC0FFEE + 1_000_003 * rank, sigma=0.02)

    # ---- device-resident throughput: W warm-up + K timed steps, CUDA events on the engine stream ----
    barrier()
    with ClockSampler(local_rank) as clocks:
        ms_total, ms_fused, launches = panel.time_device(params, warmup=args.warmup, iters=args.steps)
    barrier()
    ms_total, ms_fused = max_over_ranks(ms_total, ms_fused)
    value = units * args.steps / (ms_total * 1e-3)
    peak, peak_src = measured_peak()
    fused_ms_avg = ms_fused / args.steps
    # roofline of THIS rank's launch (the slowest rank's duration): algorithmic bytes of its own share
    achieved = ALGO_BYTES_PER_SYMBOL_BAR * S * N / (fused_ms_avg * 1e-3) / 1e9
    if args.dump_outputs and rank == 0:
        dump_outputs(panel, args.dump_outputs)
    panel.close()

    # ---- end to end through the public column API ------------------------------------------------------------------
    # One step = what a caller of the panel API does with a wide table: caller-owned f64 column buffers (ordinary
    # pageable host memory, one per {symbol}_{field}) -> pqb_suite_run_columns (thread-pool intake into pinned staging,
    # pipelined with H2D || pack + fused suite + unpack || D2H) -> pqb_panel_export_arrow (all result columns as one
    # Arrow struct array over the pinned result planes) -> release.  Timed by the host clock around the calls (they
    # return after the last D2H has landed), max over ranks.
    e2e, cpu, halted = None, None, None
    e2e_launches = 0
    if not args.no_e2e:
        import ctypes as C
        Se = min(S, args.e2e_symbols) if args.e2e_symbols else S
        threads = args.threads or max(2, min(6, (os.cpu_count() or 1) // max(world, 1)))   # (more only fights the DMA for the memory bus)
        hp = None
        while hp is None:
            try:
                hp = pq.Panel(Se, N, engine=engine, host_staging=True)
            except NV.PqbError as ex:                      # not enough page-lockable memory on this box: halve the slab
                if Se <= 1024:
                    raise
                sys.stderr.write("[bench] pinned staging for %d symbols failed (%s); halving\n" % (Se, ex))
                Se //= 2
        hp.fill_synthetic(seed=0xC0FFEE + 1_000_003 * rank, sigma=0.02, to_host=True)
        # the caller's own column buffers: copies of the panel in pageable memory, one [Se, N] matrix per field whose
        # rows are the {symbol}_{field} columns
        mats = {f: np.array(hp.host_field(f)[:Se, :N]) for f in ("close", "high", "low", "volume")}
        refs, _keep = pq.Panel.field_refs(**mats)
        arr, sch = NV.ArrowArray(), NV.ArrowSchema()
        rel_a = C.CFUNCTYPE(None, C.POINTER(NV.ArrowArray))
        rel_s = C.CFUNCTYPE(None, C.POINTER(NV.ArrowSchema))

        def step():
            hp.run_columns(refs, params, threads=threads)
            NV.check(NV.lib().pqb_panel_export_arrow(hp._h, 0, None, C.byref(arr), C.byref(sch)))
            n_cols = arr.n_children
            rel_a(arr.release)(C.pointer(arr))
            rel_s(sch.release)(C.pointer(sch))
            return n_cols

        step()                                              # warm-up (also pins / touches everything once)
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.e2e_steps):
            n_cols_out = step()
        dt = time.perf_counter() - t0
        barrier()
        (ms_host,) = max_over_ranks(dt * 1e3)
        pitch = hp.pitch
        e2e_units = Se * N * world if args.scaling == "weak" or Se != S else units
        e2e = {"value": e2e_units * args.e2e_steps / (ms_host * 1e-3), "unit": UNIT,
               "h2d_bytes_per_step": int(N_IN * Se * pitch * 8 + Se * 4),
               "d2h_bytes_per_step": int(N_OUT * Se * pitch * 8 + N_OUT * Se * hp.validity_pitch),
               "symbols_per_gpu": Se, "bars": N, "ms_per_step": ms_host / args.e2e_steps, "intake_threads_per_gpu": threads,
               "input_columns_per_gpu": int(len(refs)), "output_columns_per_gpu": int(n_cols_out),
               "timed": "host clock around pqb_suite_run_columns + pqb_panel_export_arrow, max over ranks",
               "note": "caller-owned pageable column buffers -> thread-pool intake into pinned staging || chunked H2D || "
                       "pack + fused suite + unpack || D2H -> one Arrow struct array over the pinned result planes; PCIe-bound"}
        e2e_launches = hp.last_launches() * args.e2e_steps
        # what the host <-> device link delivers on this box (all ranks at once, like the e2e step): the ceiling of the
        # e2e device -> host leg, 21 result planes out while 4 input planes come in
        gbs, perr = (C.c_double * 4)(), None
        barrier()
        try:
            NV.check(NV.lib().pqb_probe_pcie(engine._h, 2 << 30, 3, gbs))
        except Exception as ex:                             # (every rank still takes part in the collectives below)
            perr = repr(ex)
        barrier()
        lo = [-x for x in max_over_ranks(*[-g for g in gbs])]                  # the slowest rank's rates
        e2e["d2h_gbs_achieved"] = e2e["d2h_bytes_per_step"] / (e2e["ms_per_step"] * 1e-3) / 1e9
        if perr or lo[2] <= 0:
            e2e["pcie_probe"] = {"error": perr}
        else:
            e2e["pcie_probe"] = {"d2h_alone_gbs": lo[0], "h2d_alone_gbs": lo[1], "d2h_with_h2d_gbs": lo[2], "h2d_with_d2h_gbs": lo[3],
                                 "how": "pqb_probe_pcie: 2 GiB pinned <-> device copies on the engine's own streams, every rank at the "
                                        "same time, the slowest rank's rates; d2h_with_h2d_gbs bounds the e2e step's device -> host leg"}
            e2e["d2h_frac_of_link"] = e2e["d2h_gbs_achieved"] / lo[2]

        # ---- CPU baseline on rank 0: the oracle port over a bounded sample of the same panel ----
        if rank == 0 and not args.no_cpu:
            cores = os.cpu_count() or 1
            ns = min(Se, max(64, 16 * cores))
            c, h, l, v = (np.ascontiguousarray(mats[f][:ns]) for f in ("close", "high", "low", "volume"))
            rate, used, reps = cpu_suite_rate(c, h, l, v, cores, args.cpu_seconds)
            cpu = {"value": rate, "unit": UNIT, "cores": used, "kind": "port",
                   "sample": f"{ns} symbols x {N} bars of the same synthetic panel, {reps} passes, C oracle (oracle/pq_oracle.c)"}
        # ---- a realistic panel on the same staging (N = 1 only): 1 % of the symbols with a 3-bar trading halt in close,
        #      device-resident suite (engine.cu launch_suite: the blocks that hold a halted symbol run the specialised null-aware kernel
        #      -- fully valid stages take the plain steady step -- on a second stream beside the plain kernel over the other blocks) ----
        halted = None
        if world == 1 and not args.no_extra:
            try:
                n_h = max(1, Se // 100)
                okb = np.ones(N, dtype=bool)
                okb[2000:2003] = False
                bits = np.packbits(okb, bitorder="little")
                for s_ in np.linspace(0, Se - 1, n_h).astype(int):
                    hp.set_column(int(s_), "close", np.ascontiguousarray(mats["close"][int(s_)]), validity=bits)
                hp.upload()
                t_h, _, nl_h = hp.time_device(params, warmup=2, iters=5)
                halted = {"workload": "%d x %d, %d symbols (1 %%) with a 3-bar halt in close, device-resident" % (Se, N, n_h),
                          "kernel": "suite_fused_kernel<true,true> (blocks with a halted symbol, second stream) || suite_fused_kernel<true,false> "
                                    "(the other blocks) + validity", "ms": t_h / 5, "launches": nl_h,
                          "value": Se * N / (t_h / 5 * 1e-3), "unit": UNIT,
                          "vs_clean_panel": (t_h / 5) / (ms_total / args.steps) * (S / Se)}
            except Exception as ex:
                halted = {"error": repr(ex)}
        del refs, _keep, mats
        hp.close()

    # ---- the other measured shapes of BASELINE.json / SURVEY.md 8f, kernel-only, reported beside the headline
    #      (N=1 only; a few seconds each): configs 2, 3, 5, the candle kernel and the access-mix ceiling ----
    other = None
    if world == 1 and not args.no_extra:
        other = {}

        def extra(name, fn):
            try:
                other[name] = fn()
            except Exception as ex:      # never lose the headline line to an extra
                other[name] = {"error": repr(ex)}

        def c2():
            S2, N2, d2 = WORKLOADS["c2"]
            p2 = pq.Panel(S2, N2, engine=engine, host_staging=False)
            p2.fill_synthetic(seed=0xC0FFEE, sigma=0.02)
            _, f2, _ = p2.time_device(params, warmup=3, iters=20)
            p2.close()
            g2 = ALGO_BYTES_PER_SYMBOL_BAR * S2 * N2 / (f2 / 20 * 1e-3) / 1e9
            return {"workload": d2, "kernel": "suite_fused_kernel<true,false,false,true>", "kernel_ms": f2 / 20,
                    "value": S2 * N2 / (f2 / 20 * 1e-3), "unit": UNIT, "achieved_gbs": g2, "frac": g2 / peak}

        def shard8():
            # the strong-scaled shape one GPU of eight runs (6,250 symbols): what SCALE's 8-GPU point is made of
            S8 = symbol_range(WORKLOADS["c4"][0], 8, 0)[1]
            p8 = pq.Panel(S8, WORKLOADS["c4"][1], engine=engine, host_staging=False)
            p8.fill_synthetic(seed=0xC0FFEE, sigma=0.02)
            _, f8, _ = p8.time_device(params, warmup=3, iters=20)
            p8.close()
            g8 = ALGO_BYTES_PER_SYMBOL_BAR * S8 * WORKLOADS["c4"][1] / (f8 / 20 * 1e-3) / 1e9
            return {"workload": "one GPU's share of config 4 at 8 GPUs: %d x %d" % (S8, WORKLOADS["c4"][1]),
                    "kernel_ms": f8 / 20, "value": S8 * WORKLOADS["c4"][1] / (f8 / 20 * 1e-3), "unit": UNIT, "achieved_gbs": g8, "frac": g8 / peak}

        def candle():
            from polars_quant_b200 import candles
            Sc, Nc = 20_000, 5_040
            cp = candles.CandlePanel(Sc, Nc, engine=engine, host_staging=False)
            cp.fill_random_walk(seed=0xC0FFEE, sigma=0.02)
            msc = cp.time_device(warmup=3, iters=10) / 10
            cp.close()
            gc = 316 * Sc * Nc / (msc * 1e-3) / 1e9
            return {"workload": "SURVEY 8f.1: 61 cdl* patterns + 4 price transforms + bop, 20,000 x 5,040 random-walk OHLC",
                    "kernel": "candle_kernel<true>", "kernel_ms": msc, "value": Sc * Nc / (msc * 1e-3),
                    "unit": "symbol*bars/s", "algorithmic_bytes_per_symbol_bar": 316, "achieved_gbs": gc, "frac": gc / peak}

        def mix():
            # what HBM delivers for the suite's own access mix (4 planes read, 21 written, 256-byte warp rows) with no
            # arithmetic at all: the copy bandwidth used as `peak` is a 1 : 1 mix, a write-heavy stream gets less
            import ctypes as C
            msx = C.c_float()
            NV.check(NV.lib().pqb_stream_mix(engine._h, N_IN, N_OUT, 20_000 * 5_040, 2, 5, C.byref(msx)))
            gx = 8 * (N_IN + N_OUT) * 20_000 * 5_040 / (msx.value * 1e-3) / 1e9
            return {"workload": "streaming kernel, %d planes read : %d written, 20,000 x 5,040 doubles each, no arithmetic" % (N_IN, N_OUT),
                    "kernel": "stream_mix_kernel", "kernel_ms": msx.value, "achieved_gbs": gx, "frac": gx / peak,
                    "suite_over_mix": achieved / gx}

        if (S_total, N) != WORKLOADS["c2"][:2]:
            extra("c2", c2)
        extra("c4_one_of_8_gpus", shard8)
        extra("c3", lambda: bench_c3(pq, NV, engine, peak))
        extra("c5", lambda: bench_c5(pq, NV, engine, peak))
        extra("candles", candle)
        extra("access_mix_ceiling", mix)
        if not args.no_e2e and halted is not None:
            other["c4_one_percent_halted_symbols"] = halted

    if rank == 0:
        traffic, traffic_src = traffic_record(S, N)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_total / args.steps, "higher_is_better": True,
            "scaling": args.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": desc, "symbols": S_total if args.scaling == "strong" else S_total * world,
                       "symbols_per_gpu": S, "bars": N, "indicators": 15, "outputs": N_OUT,
                       "inputs": N_IN, "l2": "inputs+outputs per step (%.1f GB per GPU) are far larger than the 126 MB L2; no flush needed"
                       % (ALGO_BYTES_PER_SYMBOL_BAR * S * N / 1e9),
                       "parallelism": "symbols sharded over the GPUs in contiguous 32-symbol blocks, no collective on the data path"},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "traffic_source": traffic_src,
                         "kernel": "suite_fused_kernel<true,false>", "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": ALGO_BYTES_PER_SYMBOL_BAR * S * N,
                         "kernel_ms": fused_ms_avg, "per": "the slowest rank's launch over its own share of the panel"},
            "cpu_baseline": cpu,
            "e2e": e2e,
            "gpu_launches": launches * args.steps + e2e_launches,
            "clocks": clocks.summary(),
        }
        if other:
            line["other_workloads"] = other
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()



if __name__ == "__main__":
    main()
