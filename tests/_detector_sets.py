"""Detector parameter sets (detector_param, events.c:35-41: w_short, w_long, thr_short, thr_long, peak_height) that the
tests of sgpu_set_detector run (test infrastructure only)."""

REFERENCE = {0: (3, 6, 1.4, 9.0, 0.2), 1: (7, 14, 2.5, 9.0, 1.0)}  # events.c:43-54, chosen by rna

CUSTOM = {
    "long_below_short": (4, 9, 3.0, 1.5, 0.5),   # thr_long < thr_short: the long detector emits often
    "short_wider": (12, 5, 2.0, 2.5, 0.3),       # w_short > w_long (the reference allows it)
    "windows_2_14": (2, 14, 1.0, 3.0, 0.1),
    "windows_14_2": (14, 2, 1.5, 1.0, 0.1),
    "silent": (3, 6, 1e30, 1e30, 0.2),           # nothing is ever emitted: one event [0, n)
    "dense": (3, 2, 0.0, 0.0, 0.0),              # the most events per sample of the sets tried
    "negative_height": (3, 6, 1.0, 2.0, -0.05),  # allowed: only non-finite values are refused
}
