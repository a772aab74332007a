"""B200-native KMP packet matcher: drop-in for the hot path of Lemnon95/multithreading_string_matching.

Everything that computes lives in libkmpb200.so (C host code + sm_100a CUDA kernels, C ABI in
include/kmpb200.h); this package is the thin ctypes layer tests and bench.py drive it through."""
from ._lib import KMPB_PAT_NOCASE, KMPB_WINDOW_ANY, KMPB_WINDOW_MAX, KmpbError, LIB_PATH, SIGNATURES, lib  # noqa: F401
from .matcher import (ENGINE_AUTO, ENGINE_PERPAT, ENGINE_UNION, FIND_SORTED, MATCH_DTYPE, PROTO_TCP, PROTO_UDP,  # noqa: F401
                      SELECT_INVERT, Matcher, PayloadBatch, Synth, device_count, extract_payload, format_report,
                      load_patterns, pack_patterns, shard_range, write_selected)

__version__ = "0.1.0"
