"""The reference-facing name layer (polars_quant_b200/talib.py) against the reference's own Python shims
(python/polars_quant/talib/*.py): every shim name of the hot path and its "next" rows exists here with the same parameter
names and defaults.  Reads the reference's files from a checkout of the original named by POLARS_QUANT_REFERENCE; without
one only the committed expectations are checked."""
import inspect
import os
import re
from pathlib import Path

import pytest

from polars_quant_b200 import talib

REF = Path(os.environ.get("POLARS_QUANT_REFERENCE", ""), "python", "polars_quant", "talib")
# names the reference defines that are out of scope here (SURVEY.md section 2 / DESIGN.md section 8)
OUT_OF_SCOPE = {"HT_DCPERIOD", "HT_DCPHASE", "HT_PHASOR", "HT_SINE", "HT_TRENDLINE", "HT_TRENDMODE", "MAMA", "MAVP", "SAR", "SAREXT"}
NOT_BUILT = {"WMA", "DEMA", "T3", "KAMA", "APO", "PPO", "AROONOSC"}


def test_every_pattern_and_price_name_is_defined():
    cdl = [n for n in talib.__all__ if n.startswith("CDL")]
    assert len(cdl) == 61 and len(set(cdl)) == 61
    for n in ("AVGPRICE", "MEDPRICE", "TYPPRICE", "WCLPRICE", "BOP", "STOCHF", "STOCHRSI", "MACDEXT", "KDJ"):
        assert callable(getattr(talib, n)), n
    assert inspect.signature(talib.CDLPIERCING).parameters["penetration"].default == 0.5
    assert inspect.signature(talib.CDLMORNINGSTAR).parameters["penetration"].default == 0.3
    assert "penetration" not in inspect.signature(talib.CDLDOJI).parameters
    for n in NOT_BUILT:
        with pytest.raises(NotImplementedError):
            getattr(talib, n)(None)


@pytest.mark.skipif(not os.environ.get("POLARS_QUANT_REFERENCE") or not REF.is_dir(),
                    reason="needs POLARS_QUANT_REFERENCE: a checkout of the original polars-quant")
def test_names_parameters_and_defaults_match_the_reference_shims():
    checked = 0
    for f in sorted(REF.glob("*.py")):
        for m in re.finditer(r"^def\s+([A-Z][A-Za-z0-9_]*)\s*\(([^)]*)\)", f.read_text(), re.M):
            name, params = m.group(1), m.group(2)
            if name in OUT_OF_SCOPE:
                continue
            assert hasattr(talib, name), "%s (%s) has no counterpart" % (name, f.name)
            if name in NOT_BUILT:
                continue
            ours = inspect.signature(getattr(talib, name)).parameters
            ref_params = []
            for part in params.split(","):
                part = part.strip()
                if not part:
                    continue
                pname = part.split(":")[0].split("=")[0].strip()
                default = part.split("=")[1].strip() if "=" in part else None
                ref_params.append((pname, default))
            assert len(ours) == len(ref_params), "%s: %s vs %s" % (name, list(ours), ref_params)
            for (pname, default), (oname, op) in zip(ref_params, ours.items()):
                if default is not None:                      # keyword parameters: same name, same default
                    assert oname == pname, "%s: parameter %s vs %s" % (name, oname, pname)
                    assert float(op.default) == float(default), "%s.%s default %r vs %s" % (name, pname, op.default, default)
            checked += 1
    assert checked >= 100
