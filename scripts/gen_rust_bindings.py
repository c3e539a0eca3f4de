#!/usr/bin/env python
"""Generates the Rust `extern "C"` binding of include/pqb200.h (the block a maintainer puts in src/talib/gpu.rs of the
reference crate) so that INTEGRATION.md can never drift from the header: tests/test_integration_doc.py compares the
block inside INTEGRATION.md with this script's output.

    python scripts/gen_rust_bindings.py            # prints the block
    python scripts/gen_rust_bindings.py --write    # rewrites the block between the markers in INTEGRATION.md
"""
from __future__ import annotations

import re
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
HEADER = ROOT / "include" / "pqb200.h"
DOC = ROOT / "INTEGRATION.md"
BEGIN, END = "<!-- BEGIN GENERATED: rust bindings of include/pqb200.h -->", "<!-- END GENERATED -->"

SCALARS = {"int": "c_int", "int32_t": "i32", "int64_t": "i64", "uint32_t": "u32", "uint64_t": "u64", "double": "f64",
           "float": "f32", "uint8_t": "u8", "int8_t": "i8", "char": "c_char", "void": "c_void", "size_t": "usize"}
OPAQUE = ["pqb_engine", "pqb_panel", "pqb_multi", "pqb_candles", "pqb_split", "pqb_long", "pqb_windows", "pqb_live", "ArrowArray", "ArrowSchema"]


def camel(name: str) -> str:
    if name in ("ArrowArray", "ArrowSchema"):
        return name
    return "".join(p.capitalize() for p in name.split("_"))


def strip_comments(text: str) -> str:
    text = re.sub(r"/\*.*?\*/", " ", text, flags=re.S)
    return "\n".join(l for l in text.splitlines() if not l.lstrip().startswith("#"))      # and preprocessor lines


def rust_type(ctype: str) -> str:
    """`const pqb_col *` -> `*const PqbCol`, `pqb_panel **` -> `*mut *mut PqbPanel`, `int` -> `c_int` ..."""
    t = ctype.replace("struct ", "").strip()
    stars = t.count("*")
    base = t.replace("*", " ")
    toks = base.split()
    # `const char *const *`: a const after the first pointer level
    const_levels = []
    level_const = False
    for tok in re.findall(r"const|\*|\w+", t.replace("struct ", "")):
        if tok == "const":
            level_const = True
        elif tok == "*":
            const_levels.append(level_const)
            level_const = False
    name = [x for x in toks if x != "const"][0]
    r = SCALARS.get(name, camel(name))
    # pointer levels apply inside-out: the first `*` binds the base type
    for is_const in const_levels:
        r = ("*const " if is_const else "*mut ") + r
    return r


def parse_structs(text: str):
    out = []
    for m in re.finditer(r"typedef struct (\w+) \{(.*?)\} (\w+);", text, flags=re.S):
        fields = []
        for decl in m.group(2).split(";"):
            decl = decl.strip()
            if not decl:
                continue
            # `double pen_a, pen_b, pen_c` / `const double *values` / `int32_t reserved`
            mm = re.match(r"(.*?)([\w\s,\*]+)$", decl)
            head = decl.rsplit(" ", 1)
            first, rest = decl.split(",")[0], decl.split(",")[1:]
            tm = re.match(r"(.+?)(\**\w+)$", first.strip())
            ctype, nm = tm.group(1).strip(), tm.group(2)
            names = [nm] + [r.strip() for r in rest]
            for n in names:
                stars = n.count("*")
                fields.append((n.replace("*", ""), rust_type(ctype + " " + "*" * stars)))
        out.append((m.group(3), fields))
    return out


def parse_functions(text: str):
    out = []
    for m in re.finditer(r"PQB_API\s+(.+?)\b(pqb_\w+)\s*\((.*?)\);", text, flags=re.S):
        ret, name, params = m.group(1).strip(), m.group(2), " ".join(m.group(3).split())
        args = []
        if params and params != "void":
            for p in params.split(","):
                p = p.strip()
                am = re.match(r"(.+?)(\w+)(\[\d*\])?$", p)
                ctype, nm, arr = am.group(1).strip(), am.group(2), am.group(3)
                if arr:
                    ctype += " *"
                if nm in ("type", "in", "ref", "fn", "out", "match"):      # Rust keywords
                    nm = nm + "_"
                args.append((nm, rust_type(ctype)))
        out.append((name, args, None if ret == "void" else rust_type(ret)))
    return out


def generate() -> str:
    version = re.search(r"#define PQB_ABI_VERSION (\d+)", HEADER.read_text()).group(1)
    text = strip_comments(HEADER.read_text())
    lines = ["```rust",
             "// src/talib/gpu.rs -- GENERATED from include/pqb200.h (ABI version %s) by scripts/gen_rust_bindings.py" % version,
             "// links polars_quant_b200/libpqb200.so  (build.rs: println!(\"cargo:rustc-link-lib=dylib=pqb200\");)",
             "use std::os::raw::{c_char, c_int, c_void};",
             "pub const PQB_ABI_VERSION: c_int = %s;" % version, ""]
    for name in OPAQUE:
        lines.append("#[repr(C)] pub struct %s { _p: [u8; 0] }" % camel(name))
    lines.append("")
    for name, fields in parse_structs(text):
        lines.append("#[repr(C)]")
        lines.append("pub struct %s {" % camel(name))
        for n, t in fields:
            lines.append("    pub %s: %s," % (n, t))
        lines.append("}")
    lines.append("")
    lines.append("extern \"C\" {")
    for name, args, ret in parse_functions(text):
        sig = "    pub fn %s(%s)%s;" % (name, ", ".join("%s: %s" % a for a in args), "" if ret is None else " -> " + ret)
        lines.append(sig)
    lines.append("}")
    lines.append("```")
    return "\n".join(lines)


def doc_block() -> str:
    doc = DOC.read_text()
    a, b = doc.index(BEGIN) + len(BEGIN), doc.index(END)
    return doc[a:b].strip()


def main():
    block = generate()
    if "--write" in sys.argv:
        doc = DOC.read_text()
        a, b = doc.index(BEGIN) + len(BEGIN), doc.index(END)
        DOC.write_text(doc[:a] + "\n" + block + "\n" + doc[b:])
        print("INTEGRATION.md updated")
    else:
        print(block)


if __name__ == "__main__":
    main()
