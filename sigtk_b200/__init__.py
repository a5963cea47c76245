"""sigtk_b200 -- B200-native implementation of sigtk's per-read raw-signal hot path.

pA conversion -> Scrappie-style event detection -> per-event mean/stdv, plus the
`pa` / `stat` / `ent` / `jnn` / `prefix` siblings, as hand-written CUDA (sm_100a) behind a C-ABI
(include/sigtk_b200.h).  No CPU fallback.
"""
from ._lib import (ALIGN, EXPORTS, F_DEFAULT, F_FORCE_GENERIC, F_NO_HOST_SLOTS, F_STAGE_TIMERS, LIB_PATH, LIVE_END, LIVE_RNA,
                   LIVE_START, WANT_EVENTS, WANT_PA, WANT_STAT, WANT_ENT, WANT_JNN, WANT_PREFIX, SgpuError)
from .api import (BatchResult, Context, Detector, EventTable, ent, getevents, getevents_pa, jnn_raw, live_tables,
                  signal_in_picoamps, stat)
from . import synth

__all__ = ["ALIGN", "EXPORTS", "F_DEFAULT", "F_FORCE_GENERIC", "F_NO_HOST_SLOTS", "F_STAGE_TIMERS", "LIB_PATH", "LIVE_END", "LIVE_RNA",
           "LIVE_START", "WANT_EVENTS",
           "WANT_PA", "WANT_STAT", "WANT_ENT", "WANT_JNN", "WANT_PREFIX", "ent", "jnn_raw", "SgpuError", "BatchResult", "Context", "Detector", "EventTable", "getevents", "getevents_pa", "live_tables",
           "signal_in_picoamps", "stat", "synth"]
