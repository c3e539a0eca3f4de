"""The C oracle against the vectors made by EXECUTING the reference's own Rust / Python text
(tests/golden/talib_ref_golden.npz, generator tests/golden/make_ref_golden.py): every value bit-identical, every
validity bit identical, and the same failures (PolarsResult::Err / panic) on the same inputs.  CPU only.

This is what pins parity for SURVEY.md 8(a): the oracle is checked against outputs of the reference itself, and
the CUDA path against the oracle (tests/test_gpu_*.py) and directly against these vectors
(tests/test_gpu_ref_golden.py)."""
import collections
import os

import numpy as np
import pytest

import refgolden
from oracle import pqo

TAGS = ["A", "B", "Bs", "C3", "Cb", "D", "E0", "E1", "E2", "E10", "F", "G"]

# The oracle sees one column; a multi-chunk column is a container matter.  calc_kama's `cont_slice().unwrap()`
# (overlap.rs:826) panics on several chunks, which only the boundary could reproduce.
CHUNK_ONLY = {("C3", "kama"), ("C3", "ma_6")}


@pytest.mark.parametrize("tag", TAGS)
def test_c_oracle_reproduces_the_executed_reference(tag):
    g, index = refgolden.load()
    done = collections.Counter()
    for e in index:
        if e["tag"] != tag:
            continue
        if (tag, e["fn"]) in CHUNK_ONLY or (tag, "ma_%s" % e.get("kwargs", {}).get("matype")) in CHUNK_ONLY and e["fn"] == "ma":
            continue
        cols = refgolden.inputs(g, e)
        want = refgolden.expected(g, e)
        name = f"{tag}/{e['key']}"
        try:
            got = refgolden.oracle_call(e, cols)
        except pqo.OracleError as err:
            assert want is None, f"{name}: oracle fails ({err}) where the reference succeeds"
            # Err (1) <-> PQO_ERR_NULLS / SHAPE; panic (2) <-> PQO_ERR_PANIC.  midprice with nulls: the reference
            # dies in polars' arithmetic on unequal lengths (overlap.rs:356,401); the oracle reports it as SHAPE.
            if e["err"] == 2 and e["fn"] != "midprice":
                assert err.code == -2, f"{name}: reference panics, oracle says {err.code}"
            done["fails_alike"] += 1
            continue
        if got is None:
            done["no_oracle_entry"] += 1
            continue
        assert want is not None, f"{name}: the reference fails (err {e.get('err')}) where the oracle succeeds"
        assert len(got) == len(want), name
        for j, ((vals, ok), (gv, gok)) in enumerate(zip(got, want)):
            msg = refgolden.same(vals, ok, gv, gok)
            assert not msg, f"{name}/{j}: {msg}"
        done["bit_exact"] += 1
    assert done["bit_exact"] + done["fails_alike"] >= 90, done
    assert done["no_oracle_entry"] <= 4, done


def test_every_hot_path_function_is_pinned():
    """SURVEY.md 8(a)'s functions all appear in the golden file with at least one successful call."""
    _, index = refgolden.load()
    ok_fns = {e["fn"] for e in index if not e.get("err")}
    for fn in ("sma", "ema", "ma", "bbands", "tema", "trima", "midpoint", "midprice", "rsi", "macd", "trange", "atr",
               "natr", "obv", "ad", "adosc", "willr", "STOCH", "STOCHF", "STOCHRSI", "MACDEXT", "mom", "roc", "rocp",
               "rocr", "rocr100", "cmo", "mfi", "cci", "wma", "dema", "t3", "kama", "adx", "adxr", "dx", "plus_di",
               "minus_di", "plus_dm", "minus_dm", "trix", "ultosc", "aroon", "bop", "avgprice"):
        assert fn in ok_fns, fn


def test_first_valid_index_contract_of_the_reference():
    """SURVEY.md 8a's "first non-null index" table, read off the reference's own outputs (case A, 1 x 252)."""
    g, _ = refgolden.load()
    first = lambda key: int(np.argmax(g[key]))
    assert first("A/sma_30/0/ok") == 29 and first("A/ema_30/0/ok") == 29
    assert first("A/tema_30/0/ok") == 87 and first("A/trima_30/0/ok") == 29
    assert first("A/bbands_20/0/ok") == 19
    assert first("A/macd_12_26_9/0/ok") == 25 and first("A/macd_12_26_9/1/ok") == 8 and first("A/macd_12_26_9/2/ok") == 25
    assert np.all(g["A/macd_12_26_9/1/v"][8:25] == 0.0)           # zero-filled signal warm-up (momentum.rs:268-271)
    assert first("A/rsi_14/0/ok") == 13 and first("A/trange/0/ok") == 1
    assert first("A/atr_default/0/ok") == 27 and first("A/natr_14/0/ok") == 27
    assert first("A/obv/0/ok") == 1 and first("A/ad/0/ok") == 0 and first("A/adosc_3_10/0/ok") == 9
    assert first("A/willr_14/0/ok") == 13 and first("A/midpoint_14/0/ok") == 0 and first("A/midprice_14/0/ok") == 0
    assert first("A/STOCH_9_3_3/0/ok") == 10 and first("A/STOCH_9_3_3/1/ok") == 12
    assert first("A/STOCHF_5_3/0/ok") == 4


@pytest.mark.skipif(not os.environ.get("POLARS_QUANT_REFERENCE") or
                    not os.path.isdir(os.path.join(os.environ["POLARS_QUANT_REFERENCE"], "src", "talib")),
                    reason="needs POLARS_QUANT_REFERENCE: a checkout of the original polars-quant")
def test_golden_file_is_what_the_reference_text_produces_today():
    """Re-executes a sample of the calls from the original's source text and compares with the committed file (provenance)."""
    import sys
    sys.path.insert(0, str(refgolden.ROOT / "tests" / "golden"))
    from rustexec.ref_exec import Reference, series
    g, index = refgolden.load()
    ref = Reference()
    n = 0
    for e in index:
        if e["tag"] not in ("A", "B") or e["kind"] != "rs" or e.get("err"):
            continue
        cols = refgolden.inputs(g, e)
        res = ref.call(e["fn"], [series(*cols[c]) for c in e["cols"]], e["params"], e["kwargs"])
        for (vals, ok), (gv, gok) in zip(res, refgolden.expected(g, e)):
            assert not refgolden.same(vals, ok, gv, gok), e["key"]
        n += 1
    assert n > 100
