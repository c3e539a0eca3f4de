import os
from pathlib import Path


def reference_root() -> Path:
    """Root of a checkout of the original polars-quant (src/talib/*.rs, python/polars_quant/).  Nothing of it is stored
    in this repository; the golden-vector generators and the provenance tests read it from POLARS_QUANT_REFERENCE."""
    root = os.environ.get("POLARS_QUANT_REFERENCE")
    if not root:
        raise RuntimeError("set POLARS_QUANT_REFERENCE to a checkout of the original polars-quant")
    return Path(root)
