"""Live screens without a GPU: the C ABI refuses to create one (no CPU fallback), the Python screen argument is checked
on the host, the header documents the rules, and the ctypes mirror of pqb_live_screen matches the header."""
import ctypes as C
import re
import subprocess
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parents[1]


@pytest.fixture(scope="module")
def N():
    from polars_quant_b200 import _native as N
    N.build()
    return N


def test_create_without_a_device_is_no_device(N):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    scr = N.LiveScreen()
    N.lib().pqb_live_screen_default(C.byref(scr))
    out = C.c_void_p()
    rc = N.lib().pqb_live_create_screen(None, C.byref(N.default_params()), 0, 64, 0, C.byref(scr), C.byref(out))
    assert rc == -1 and not out.value                     # PQB_ERR_NO_DEVICE
    assert b"no CPU fallback" in N.lib().pqb_last_error()
    assert not N.lib().pqb_live_host_signal(None, 0) and not N.lib().pqb_live_host_info(None)
    assert not N.lib().pqb_live_host_info_valid(None)
    assert N.lib().pqb_live_info(None, None, None) == -3   # PQB_ERR_INVALID


def test_the_python_defaults_are_the_c_defaults(N):
    from polars_quant_b200.live import screen_struct
    want = N.LiveScreen()
    N.lib().pqb_live_screen_default(C.byref(want))
    got = screen_struct(True)
    assert [getattr(got, f) for f, _ in N.LiveScreen._fields_] == [getattr(want, f) for f, _ in N.LiveScreen._fields_]
    assert (want.oversold, want.overbought, want.ma_type, want.ma_fast, want.ma_slow, want.info) == (30.0, 70.0, 0, 10, 20, 1)
    assert screen_struct(None) is None and screen_struct(False) is None
    s = screen_struct(dict(oversold=25, overbought=80, ma_cross=("ema", 5, 60), info=False))
    assert (s.oversold, s.overbought, s.ma_type, s.ma_fast, s.ma_slow, s.info) == (25.0, 80.0, 1, 5, 60, 0)
    assert screen_struct(dict(ma_cross=None)).ma_type == -1


@pytest.mark.parametrize("bad, exc", [
    ("yes", TypeError),
    (dict(oversold=30, ma=("sma", 10, 20)), ValueError),           # unknown key
    (dict(ma_cross=("wma", 10, 20)), ValueError),                  # not built
    (dict(ma_cross=("sma", 10)), ValueError),                      # two of three
    (dict(ma_cross="sma"), ValueError),
    (dict(ma_cross=("sma", 10.5, 20)), TypeError),
    (dict(info="yes"), TypeError),
])
def test_screen_argument_errors(N, bad, exc):
    from polars_quant_b200.live import screen_struct
    with pytest.raises(exc):
        screen_struct(bad)


def test_info_needs_a_screen_on_a_shell_object(N):
    from polars_quant_b200.live import LivePanel
    lp = LivePanel.__new__(LivePanel)
    lp.n_symbols, lp.max_push_bars, lp._h, lp.outputs = 5, 4, None, []
    with pytest.raises(ValueError, match="screen info"):
        lp.info()
    assert lp.signals == {} and lp.last_info == {}


def _section():
    text = (ROOT / "include" / "pqb200.h").read_text()
    a = text.index("---- live screens")
    lines = text[a:text.index("PQB_API int pqb_live_info", a)].splitlines()
    return " ".join(" ".join(re.sub(r"^\s*\*\s?", "", ln) for ln in lines).split())


def test_header_section_names_the_rules():
    s = _section()
    for phrase in ("a null on either bar gives 0", "pqb_signals_run", "pqb_ma_cross_run", "pqb_panel_info",
                   "PQB_ERR_UNSUPPORTED at create", "A preview (commit = 0) returns its signals and info and keeps nothing",
                   "symbols that start inside a push", "validity exactly", "pqb_live_info()"):
        assert phrase in s, phrase
    assert re.search(r"PQB_LIVE_NULLS panel asking for ma_type >= 0 or info is PQB_ERR_UNSUPPORTED", s)


def test_ctypes_mirror_matches_the_header(N, tmp_path):
    import sys
    sys.path.insert(0, str(ROOT / "scripts"))
    import gen_rust_bindings as G
    text = G.strip_comments(G.HEADER.read_text())
    body = re.search(r"typedef struct pqb_live_screen \{(.*?)\} pqb_live_screen;", text, flags=re.S).group(1)
    names = []
    for decl in body.split(";"):
        decl = " ".join(decl.split())
        if decl:
            ctype, rest = re.match(r"(\w+)\s+(.*)", decl).groups()
            names += [(n.strip(), ctype) for n in rest.split(",")]
    ct = {"double": C.c_double, "int32_t": C.c_int32}
    assert [(n, ct[t]) for n, t in names] == list(N.LiveScreen._fields_)
    src = '#include "%s"\n#include <stdio.h>\n#include <stddef.h>\nint main(void){printf("%%zu %%zu", sizeof(pqb_live_screen), offsetof(pqb_live_screen, info));return 0;}' % G.HEADER
    exe = tmp_path / "sizes.out"
    subprocess.run(["gcc", "-x", "c", "-", "-o", str(exe)], input=src.encode(), check=True)
    size, off = (int(x) for x in subprocess.run([str(exe)], capture_output=True, check=True).stdout.split())
    assert (size, off) == (C.sizeof(N.LiveScreen), N.LiveScreen.info.offset)
