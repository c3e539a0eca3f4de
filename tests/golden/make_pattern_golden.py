#!/usr/bin/env python
"""Golden vectors for the 61 candlestick patterns + price transforms + BOP (SURVEY.md 8f.1), made by
EXECUTING the reference's own Rust text.

The reference cannot be compiled in this image (no cargo/rustc), but src/talib/pattern.rs is written in
a tiny, regular subset of Rust: per function one `for i in K..n { let x = <expr>; ... if m { out[i] = V; } }`
loop over plain f64 comparisons, plus a dozen one-line helper predicates.  This script translates that
text to Python MECHANICALLY, token for token (`&&` -> `and`, `||` -> `or`, `let` dropped, braces ->
indentation, `(a).abs()` -> `abs(a)`, `a.min(b)` -> `min(a, b)`), at generation time, from a checkout
of the original, and runs it on the candle panel below -- so the vectors are the reference's own
arithmetic (Python floats are IEEE f64, comparisons identical), not a hand restatement.  Nothing of the
translated source is stored: only this script, the seeds and the outputs travel.  Python's
`min`/`max` differ from Rust's f64::min/max only for NaN operands; the panel has none.

usage (POLARS_QUANT_REFERENCE set to a checkout of the original polars-quant):
    python tests/golden/make_pattern_golden.py            # writes tests/golden/candle_golden.npz
"""
from __future__ import annotations

import re
import sys
from pathlib import Path

import numpy as np

from rustexec import reference_root

REF = reference_root() / "src" / "talib"
OUT = Path(__file__).resolve().parent / "candle_golden.npz"


# ---------------------------------------------------------------------------------------------------
# the candle panel: 48 symbols x 400 bars on a coarse price grid (so equalities, dojis, gaps and
# marubozus occur), a few regimes of body / shadow size so that every pattern family fires
# ---------------------------------------------------------------------------------------------------
def candle_panel(n_symbols: int = 48, n_bars: int = 400, seed: int = 20260117):
    rng = np.random.Generator(np.random.Philox(seed))
    o = np.empty((n_symbols, n_bars)); h = np.empty_like(o); l = np.empty_like(o); c = np.empty_like(o)
    for s in range(n_symbols):
        tick = [0.01, 0.05, 0.25, 0.5][s % 4]
        price = 20.0 + 5.0 * (s % 7)
        regime = s % 6
        prev_c = price
        run = 0
        for t in range(n_bars):
            if run == 0:
                trend = rng.choice([-1, 0, 1])
                run = int(rng.integers(2, 7))
            run -= 1
            gap = rng.choice([0.0, 0.0, 0.0, 1.0, -1.0, 2.0, -2.0]) * price * 0.01 * (1 + regime)
            op = prev_c + gap
            big = [0.02, 0.06, 0.10, 0.04, 0.08, 0.12][regime]
            kind = rng.integers(0, 10)
            if kind < 2:
                body = 0.0                                             # doji
            elif kind < 5:
                body = price * rng.uniform(0.0, 0.02)                  # short body
            else:
                body = price * rng.uniform(0.03, big + 0.03)           # long body
            sign = trend if trend != 0 and rng.random() < 0.75 else rng.choice([-1, 1])
            cl = op + sign * body
            sh = rng.integers(0, 6)
            up = price * [0.0, 0.0, 0.002, 0.02, 0.08, 0.15][sh]
            sh = rng.integers(0, 6)
            dn = price * [0.0, 0.0, 0.002, 0.02, 0.08, 0.15][sh]
            hi = max(op, cl) + up
            lo = min(op, cl) - dn
            q = lambda x: max(tick, round(x / tick) * tick)
            op, cl, hi, lo = q(op), q(cl), q(hi), q(lo)
            hi = max(hi, op, cl); lo = min(lo, op, cl)
            o[s, t], h[s, t], l[s, t], c[s, t] = op, hi, lo, cl
            prev_c = cl
            price = max(5.0, cl)
    return o, h, l, c


# ---------------------------------------------------------------------------------------------------
# mechanical Rust -> Python translation of pattern.rs
# ---------------------------------------------------------------------------------------------------
HELPERS: set = set()


def _expr(e: str) -> str:
    e = e.replace("&&", " and ").replace("||", " or ")
    # Rust lets `let long_body = long_body(o, c);` shadow the helper; Python does not: helpers get a prefix
    e = re.sub(r"\b(%s)\(" % "|".join(sorted(HELPERS)), r"H_\1(", e) if HELPERS else e
    e = re.sub(r"!\s*(?=[A-Za-z_(])", " not ", e)
    # method calls of the helper section
    for _ in range(8):
        e2 = re.sub(r"\(([^()]*)\)\.abs\(\)", r"abs(\1)", e)
        e2 = re.sub(r"\b([A-Za-z_]\w*)\.min\(([^()]*)\)", r"min(\1, \2)", e2)
        e2 = re.sub(r"\b([A-Za-z_]\w*)\.max\(([^()]*)\)", r"max(\1, \2)", e2)
        if e2 == e:
            break
        e = e2
    return e


def translate_pattern_rs(text: str) -> str:
    py = ["def _out(n):\n    return [0] * n\n"]
    # statements: join physical lines until ';', '{' or '}' closes one
    body_start = text.index("pub fn")
    stmts, cur = [], ""
    for raw in text[body_start:].splitlines():
        t = raw.strip()
        if not t or t.startswith("//") or t.startswith("#["):
            continue
        cur = (cur + " " + t).strip()
        if cur.endswith((";", "{", "}")):
            stmts.append(cur)
            cur = ""
    depth = 0
    skip_until_semicolon = False
    for s in stmts:
        ind = "    " * depth
        if s.startswith("pub fn ") or s.startswith("fn "):
            m = re.match(r"(?:pub )?fn (\w+)\((.*?)\)(?: -> .*?)? \{", s)
            name, args = m.group(1), m.group(2)
            if "inputs" in args:
                py.append(f"\ndef {name}(open, high, low, close, penetration_arg=None):")
                py.append("    n = len(open)")
                py.append("    out = _out(n)")
            else:
                names = [a.split(":")[0].strip() for a in args.split(",")]
                py.append(f"\ndef {name}({', '.join(names)}):")
            depth = 1
            continue
        if s == "}":
            depth -= 1
            continue
        m = re.match(r"\} else if (.*) \{", s)
        if m:
            py.append("    " * (depth - 1) + f"elif {_expr(m.group(1))}:")
            continue
        if s == "} else {":
            py.append("    " * (depth - 1) + "else:")
            continue
        m = re.match(r"for (\w+) in (\w+)\.\.(\w+) \{", s)
        if m:
            py.append(ind + f"for {m.group(1)} in range({m.group(2)}, {m.group(3)}):")
            depth += 1
            continue
        m = re.match(r"if (.*) \{", s)
        if m:
            py.append(ind + f"if {_expr(m.group(1))}:")
            depth += 1
            continue
        if re.match(r"let (open|high|low|close) = ", s) or s in ("let n = open.len();", "let mut out = vec![0i32; n];"):
            continue
        m = re.match(r"let penetration = inputs \.get\(4\) \.and_then\(\|s\| s\.f64\(\)\.ok\(\)\?\.get\(0\)\) \.unwrap_or\(([\d.]+)\);", s)
        if m:
            py.append(ind + f"penetration = {m.group(1)} if penetration_arg is None else penetration_arg")
            continue
        if s.startswith("Ok(Int32Chunked"):
            py.append(ind + "return out")
            continue
        m = re.match(r"let (?:mut )?(\w+) = (.*);", s)
        if m:
            py.append(ind + f"{m.group(1)} = {_expr(m.group(2))}")
            continue
        m = re.match(r"(out\[\w+\]) = (-?\d+);", s)
        if m:
            py.append(ind + f"{m.group(1)} = {m.group(2)}")
            continue
        if depth >= 1 and not s.endswith(("{", "}")) and s.endswith(";") is False:
            pass
        # helper bodies are single expressions without ';'
        raise SystemExit(f"untranslated statement: {s!r}")
    return "\n".join(py) + "\n"


def load_reference_patterns():
    text = (REF / "pattern.rs").read_text()
    # helper predicates end without ';' (expression bodies): give them one so the statement splitter sees them
    head, aux = text.split("// --- Auxiliary Functions ---", 1)
    aux = aux.replace("// --- Auxiliary Functions ---", "")
    aux_py = []
    found = list(re.finditer(r"fn (\w+)\((.*?)\) -> (?:bool|f64) \{\s*(.*?)\s*\}", aux, flags=re.S))
    HELPERS.update(m.group(1) for m in found)
    for m in found:
        names = [a.split(":")[0].strip() for a in m.group(2).split(",")]
        aux_py.append(f"def H_{m.group(1)}({', '.join(names)}):\n    return {_expr(' '.join(m.group(3).split()))}\n")
    src = "\n".join(aux_py) + translate_pattern_rs(head)
    ns: dict = {}
    exec(compile(src, "<pattern.rs translated>", "exec"), ns)
    names = re.findall(r"pub fn (cdl\w+)\(", head)
    return names, ns


def price_and_bop(o, h, l, c):
    """price.rs:10-91 and momentum.rs:113-135, evaluated with Python floats in the source's operation order."""
    n = len(o)
    avg = [(o[i] + h[i] + l[i] + c[i]) * 0.25 for i in range(n)]
    med = [(h[i] + l[i]) * 0.5 for i in range(n)]
    typ = [(h[i] + l[i] + c[i]) / 3.0 for i in range(n)]
    wcl = [(h[i] + l[i] + 2.0 * c[i]) / 4.0 for i in range(n)]
    bop = [0.0 if (h[i] - l[i]) == 0.0 else (c[i] - o[i]) / (h[i] - l[i]) for i in range(n)]
    return avg, med, typ, wcl, bop


def search_window(f, rng, tries: int = 400_000):
    """Random search for a 6-bar window on which pattern `f` fires (for the patterns too rare for the panel)."""
    for _ in range(tries):
        p = 50.0
        prev_o, prev_c = p, p * (1 + rng.choice([-0.08, 0.08]))
        O, H, L, C = [], [], [], []
        for k in range(6):
            lo_b, hi_b = min(prev_o, prev_c), max(prev_o, prev_c)
            where = rng.integers(0, 7)
            op = [hi_b * 1.03, lo_b * 0.97, rng.uniform(lo_b, hi_b), prev_c, prev_o, hi_b * 1.005, lo_b * 0.995][where]
            kind = rng.integers(0, 6)
            body = op * [0.0, 0.01, 0.03, 0.07, 0.12, 0.2][kind]
            cl = op + rng.choice([-1.0, 1.0]) * body
            up = op * [0.0, 0.0005, 0.01, 0.05, 0.2][rng.integers(0, 5)]
            dn = op * [0.0, 0.0005, 0.01, 0.05, 0.2][rng.integers(0, 5)]
            O.append(op); C.append(cl); H.append(max(op, cl) + up); L.append(min(op, cl) - dn)
            prev_o, prev_c = op, cl
        out = f(O, H, L, C)
        if any(out):
            return O, H, L, C
    return None


def main():
    names, ns = load_reference_patterns()
    assert len(names) == 61, len(names)
    o, h, l, c = candle_panel()
    # plant windows for the patterns the random panel never produces (two extra symbols)
    rng = np.random.Generator(np.random.Philox(77))
    rare = []
    for name in names:
        fired = any(any(ns[name](o[s].tolist(), h[s].tolist(), l[s].tolist(), c[s].tolist())) for s in range(o.shape[0]))
        if not fired:
            rare.append(name)
    extra = [np.repeat(x[:2], 1, axis=0).copy() for x in (o, h, l, c)]
    pos = 10
    for name in rare:
        for rep in range(2):
            w = search_window(ns[name], rng)
            if w is None:
                print("no window found for", name)
                break
            for x, col in zip(extra, w):
                x[rep, pos:pos + 6] = col
            pos += 9
    o, h, l, c = (np.concatenate([x, e], axis=0) for x, e in zip((o, h, l, c), extra))
    S, N = o.shape
    pat = np.zeros((len(names), S, N), dtype=np.int16)
    for k, name in enumerate(names):
        f = ns[name]
        for s in range(S):
            pat[k, s] = f(o[s].tolist(), h[s].tolist(), l[s].tolist(), c[s].tolist())
    hits = {n: (int((pat[k] > 0).sum()), int((pat[k] < 0).sum())) for k, n in enumerate(names)}
    never = [n for n, (a, b) in hits.items() if a + b == 0]
    print("patterns that never fire on the panel:", never)
    for n, (a, b) in hits.items():
        print(f"  {n:24s} +{a:5d} -{b:5d}")
    # a second penetration value for the five functions that take one
    pen_names = [n for n in names if "penetration" in (REF / "pattern.rs").read_text().split("pub fn " + n + "(")[1].split("pub fn ")[0]]
    pen = np.zeros((len(pen_names), S, N), dtype=np.int16)
    for k, name in enumerate(pen_names):
        for s in range(S):
            pen[k, s] = ns[name](o[s].tolist(), h[s].tolist(), l[s].tolist(), c[s].tolist(), 0.55)
    prices = np.zeros((5, S, N))
    for s in range(S):
        for k, col in enumerate(price_and_bop(o[s].tolist(), h[s].tolist(), l[s].tolist(), c[s].tolist())):
            prices[k, s] = col
    np.savez_compressed(OUT, names=np.array(names), open=o, high=h, low=l, close=c, patterns=pat,
                        penetration_names=np.array(pen_names), penetration_value=np.array(0.55), patterns_pen=pen,
                        prices=prices, price_names=np.array(["avgprice", "medprice", "typprice", "wclprice", "bop"]))
    print("wrote", OUT, OUT.stat().st_size, "bytes")
    # cdl2crows can never fire in the reference: `open_in2 = (o > o2) && (o < c2)` (pattern.rs:31) contradicts
    # `bear2 = bear(o2, c2)` (c2 < o2); its golden column is all zeros
    return 1 if set(never) - {"cdl2crows"} else 0


if __name__ == "__main__":
    sys.exit(main())
