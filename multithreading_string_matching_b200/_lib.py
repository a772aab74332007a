"""ctypes binding of libkmpb200.so (include/kmpb200.h).  The library is built in-tree by
`make -C multithreading_string_matching_b200` (or __graft_entry__.build()); there is no Python or CPU
fallback: importing this module without the shared library raises."""
import ctypes
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libkmpb200.so")

c_u8p = ctypes.POINTER(ctypes.c_uint8)
c_u32p = ctypes.POINTER(ctypes.c_uint32)
c_u64p = ctypes.POINTER(ctypes.c_uint64)
c_i32p = ctypes.POINTER(ctypes.c_int32)

KMPB_PAT_NOCASE = 1  # kmpb_set_patterns_ex: ASCII case-insensitive pattern
KMPB_WINDOW_ANY = 0xFFFFFFFF  # kmpb_set_patterns_win: {0, KMPB_WINDOW_ANY} is no window
KMPB_WINDOW_MAX = 65535  # the largest hi of a window


class KmpbError(RuntimeError):
    def __init__(self, code, message):
        super().__init__("libkmpb200 error %d: %s" % (code, message))
        self.code = code


class CPatterns(ctypes.Structure):
    _fields_ = [("blob", c_u8p), ("pat_off", c_u32p), ("n_pat", ctypes.c_uint32)]


class CCsr(ctypes.Structure):
    _fields_ = [("bytes", c_u8p), ("offsets", c_u64p), ("n_packets", ctypes.c_uint64),
                ("n_frames", ctypes.c_uint64), ("total_bytes", ctypes.c_uint64), ("pinned", ctypes.c_int)]


class CWindow(ctypes.Structure):
    _fields_ = [("lo", ctypes.c_uint32), ("hi", ctypes.c_uint32)]


class CSynth(ctypes.Structure):
    _fields_ = [("seed", ctypes.c_uint64), ("payload_len", ctypes.c_uint32), ("len_mode", ctypes.c_uint32),
                ("plants", ctypes.c_uint32), ("plant_blob", c_u8p), ("plant_off", c_u32p),
                ("n_plant", ctypes.c_uint32)]


# name -> (restype, argtypes): every symbol include/kmpb200.h declares
SIGNATURES = {
    "kmpb_version": (ctypes.c_char_p, []),
    "kmpb_last_error": (ctypes.c_char_p, []),
    "kmpb_device_count": (ctypes.c_int, []),
    "kmpb_device_ordinal": (ctypes.c_int, [ctypes.c_int]),
    "kmpb_check_device_errors": (ctypes.c_int, [ctypes.c_void_p]),
    "kmpb_create": (ctypes.c_int, [ctypes.POINTER(ctypes.c_void_p), ctypes.c_int]),
    "kmpb_destroy": (None, [ctypes.c_void_p]),
    "kmpb_set_engine": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int]),
    "kmpb_get_device": (ctypes.c_int, [ctypes.c_void_p]),
    "kmpb_set_patterns": (ctypes.c_int, [ctypes.c_void_p, c_u8p, c_u32p, ctypes.c_uint32]),
    "kmpb_set_patterns_ex": (ctypes.c_int, [ctypes.c_void_p, c_u8p, c_u32p, ctypes.c_uint32, c_u8p]),
    "kmpb_set_patterns_win": (ctypes.c_int, [ctypes.c_void_p, c_u8p, c_u32p, ctypes.c_uint32, c_u8p,
                                             ctypes.POINTER(CWindow)]),
    "kmpb_pattern_count": (ctypes.c_uint32, [ctypes.c_void_p]),
    "kmpb_get_prefix": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_uint32, c_i32p, ctypes.c_uint32]),
    "kmpb_count_host": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint64, c_u64p]),
    "kmpb_count_device": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint64,
                                         ctypes.c_void_p, ctypes.c_void_p]),
    "kmpb_count_device_span": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint64,
                                              ctypes.c_uint64, ctypes.c_uint64, ctypes.c_void_p, ctypes.c_void_p]),
    "kmpb_count_device_span_peers": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint64,
                                                   ctypes.c_uint64, ctypes.c_uint64, ctypes.POINTER(ctypes.c_void_p),
                                                   ctypes.c_uint32, ctypes.c_void_p]),
    "kmpb_device_counts": (ctypes.c_void_p, [ctypes.c_void_p]),
    "kmpb_set_profile": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int]),
    "kmpb_last_kernel_ms": (ctypes.c_int, [ctypes.c_void_p, ctypes.POINTER(ctypes.c_double)]),
    "kmpb_launch_count": (ctypes.c_uint64, [ctypes.c_void_p]),
    "kmpb_last_timing": (ctypes.c_int, [ctypes.c_void_p, ctypes.POINTER(ctypes.c_double), ctypes.c_int]),
    "kmpb_shard_range": (None, [ctypes.c_uint64, ctypes.c_uint32, ctypes.c_uint32, c_u64p, c_u64p]),
    "kmpb_host_alloc": (ctypes.c_void_p, [ctypes.c_size_t]),
    "kmpb_host_free": (None, [ctypes.c_void_p]),
    "kmpb_extract_udp": (ctypes.c_int, [c_u8p, ctypes.c_uint32, c_u32p, c_u32p]),
    "kmpb_extract_tcp": (ctypes.c_int, [c_u8p, ctypes.c_uint32, c_u32p, c_u32p]),
    "kmpb_load_patterns_file": (ctypes.c_int, [ctypes.c_char_p, ctypes.POINTER(CPatterns)]),
    "kmpb_free_patterns": (None, [ctypes.POINTER(CPatterns)]),
    "kmpb_load_pcap_csr": (ctypes.c_int, [ctypes.c_char_p, ctypes.c_int, ctypes.c_int, ctypes.POINTER(CCsr)]),
    "kmpb_free_csr": (None, [ctypes.POINTER(CCsr)]),
    "kmpb_pcap_open": (ctypes.c_int, [ctypes.c_char_p, ctypes.c_int, ctypes.POINTER(ctypes.c_void_p)]),
    "kmpb_pcap_close": (None, [ctypes.c_void_p]),
    "kmpb_pcap_packets": (ctypes.c_uint64, [ctypes.c_void_p]),
    "kmpb_pcap_frames": (ctypes.c_uint64, [ctypes.c_void_p]),
    "kmpb_pcap_bytes": (ctypes.c_uint64, [ctypes.c_void_p]),
    "kmpb_count_pcap": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint64, ctypes.c_uint64, c_u64p]),
    "kmpb_reserve_staging": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_uint64, ctypes.c_uint64]),
    "kmpb_find_device_span": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint64,
                                             ctypes.c_uint64, ctypes.c_uint64, ctypes.c_void_p, ctypes.c_uint64,
                                             ctypes.c_void_p, ctypes.c_uint32, ctypes.c_void_p]),
    "kmpb_find_host": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint64,
                                      ctypes.c_void_p, ctypes.c_uint64, c_u64p]),
    "kmpb_find_pcap": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint64, ctypes.c_uint64,
                                      ctypes.c_void_p, ctypes.c_uint64, c_u64p]),
    "kmpb_select_device_span": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint64,
                                               ctypes.c_uint64, ctypes.c_uint64, ctypes.c_void_p, ctypes.c_void_p,
                                               ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint32, ctypes.c_void_p]),
    "kmpb_select_host": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint64,
                                        ctypes.c_void_p, c_u64p, ctypes.c_void_p]),
    "kmpb_select_pcap": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint64, ctypes.c_uint64,
                                        ctypes.c_void_p, c_u64p, ctypes.c_void_p]),
    "kmpb_pcap_write_selected": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_uint64, ctypes.c_uint64, ctypes.c_void_p,
                                                ctypes.c_int, ctypes.c_char_p, c_u64p]),
    "kmpb_pcap_frame_index": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_uint64, ctypes.c_uint64, ctypes.c_void_p]),
    "kmpb_stream_open": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.c_uint64, ctypes.POINTER(ctypes.c_void_p)]),
    "kmpb_stream_push": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_char_p, ctypes.c_uint32]),
    "kmpb_stream_flush": (ctypes.c_int, [ctypes.c_void_p, c_u64p]),
    "kmpb_stream_packets": (ctypes.c_uint64, [ctypes.c_void_p]),
    "kmpb_stream_close": (None, [ctypes.c_void_p]),
    "kmpb_print_report": (ctypes.c_int, [ctypes.c_void_p, ctypes.POINTER(CPatterns), c_u64p]),
    "kmpb_synth_bytes": (ctypes.c_uint64, [ctypes.POINTER(CSynth), ctypes.c_uint64, ctypes.c_uint64]),
    "kmpb_synth_fill_host": (ctypes.c_int, [ctypes.POINTER(CSynth), ctypes.c_uint64, ctypes.c_uint64,
                                            ctypes.c_void_p, ctypes.c_void_p]),
    "kmpb_synth_fill_device": (ctypes.c_int, [ctypes.c_void_p, ctypes.POINTER(CSynth), ctypes.c_uint64,
                                              ctypes.c_uint64, ctypes.c_void_p, ctypes.c_void_p]),
}

_lib = None


def lib():
    """The loaded shared library; raises when it has not been built (no fallback of any kind)."""
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise ImportError("%s is missing: build it with `make -C %s` (python -c 'import __graft_entry__ as g; "
                              "g.build()'); this package has no CPU or PyTorch fallback" % (LIB_PATH, HERE))
        L = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)  # AttributeError here means header and library disagree
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(rc):
    if rc != 0:
        raise KmpbError(rc, lib().kmpb_last_error().decode("utf-8", "replace"))
