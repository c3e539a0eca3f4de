"""INTEGRATION.md's Rust binding, the C header and the ctypes mirror must describe the same ABI (round-1 verdict: the
hand-written Rust block had drifted -- u32 outputs_mask, seven missing pqb_suite_params fields).  CPU only."""
import ctypes as C
import re
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT / "scripts"))
import gen_rust_bindings as G  # noqa: E402

CTYPES = {"int": C.c_int, "int32_t": C.c_int32, "int64_t": C.c_int64, "uint32_t": C.c_uint32, "uint64_t": C.c_uint64,
          "double": C.c_double, "float": C.c_float}


def header_struct(name):
    text = G.strip_comments(G.HEADER.read_text())
    m = re.search(r"typedef struct %s \{(.*?)\} %s;" % (name, name), text, flags=re.S)
    fields = []
    for decl in m.group(1).split(";"):
        decl = " ".join(decl.split())
        if not decl:
            continue
        tm = re.match(r"(.+?)\s*(\**\w+(?:\s*,\s*\**\w+)*)$", decl)
        ctype, names = tm.group(1).strip(), [n.strip() for n in tm.group(2).split(",")]
        for n in names:
            fields.append((n.replace("*", ""), ctype + (" *" if "*" in n else "")))
    return fields


def test_integration_md_carries_the_generated_binding():
    assert G.doc_block() == G.generate().strip(), "run: python scripts/gen_rust_bindings.py --write"


def test_generated_binding_covers_every_declared_function_and_struct_field():
    text = G.strip_comments(G.HEADER.read_text())
    block = G.generate()
    for fn in set(re.findall(r"PQB_API\s+[\w\s\*]+?\b(pqb_\w+)\s*\(", text)):
        assert "pub fn %s(" % fn in block, fn
    for struct in ("pqb_suite_params", "pqb_col_ref", "pqb_col", "pqb_out_col", "pqb_candle_params"):
        for name, _ in header_struct(struct):
            assert re.search(r"pub %s: " % name, block), (struct, name)
    assert "outputs_mask: u64" in block and "pub donchian_period: i32" in block


def test_ctypes_mirror_matches_the_header_layouts(tmp_path):
    from polars_quant_b200 import _native as N
    for struct, mirror in (("pqb_suite_params", N.SuiteParams), ("pqb_col_ref", N.ColRef), ("pqb_col", N.Col),
                           ("pqb_out_col", N.OutCol), ("pqb_candle_params", N.CandleParams)):
        want = header_struct(struct)
        got = list(mirror._fields_)
        assert [n for n, _ in want] == [n for n, _ in got], struct
        for (name, ctype), (_, ct) in zip(want, got):
            if "*" in ctype:
                assert ct is C.c_void_p, (struct, name)
            else:
                assert ct is CTYPES[ctype.replace("const ", "")], (struct, name, ctype)
    # and the sizes the C compiler gives the same structs
    src = '#include "%s"\n#include <stdio.h>\nint main(void){printf("%%zu %%zu %%zu %%zu %%zu", sizeof(pqb_suite_params), sizeof(pqb_col_ref), sizeof(pqb_col), sizeof(pqb_out_col), sizeof(pqb_candle_params));return 0;}' % G.HEADER
    exe = tmp_path / "sizes.out"
    subprocess.run(["gcc", "-x", "c", "-", "-o", str(exe)], input=src.encode(), check=True)
    sizes = [int(x) for x in subprocess.run([str(exe)], capture_output=True, check=True).stdout.split()]
    assert sizes == [C.sizeof(N.SuiteParams), C.sizeof(N.ColRef), C.sizeof(N.Col), C.sizeof(N.OutCol), C.sizeof(N.CandleParams)]
