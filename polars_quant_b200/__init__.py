"""polars_quant_b200 -- B200-native drop-in for polars-quant's src/talib indicator engine on
wide `{symbol}_{column}` f64 panels.  CUDA (sm_100a) behind a C ABI; no CPU fallback."""
from . import _native
from .panel import Engine, MultiPanel, Panel, SplitPanel, get_engine
from .live import LivePanel
from . import shard

__all__ = ["Engine", "LivePanel", "MultiPanel", "Panel", "SplitPanel", "get_engine", "shard", "_native"]
