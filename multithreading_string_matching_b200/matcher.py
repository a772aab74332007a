"""Host-side mirror of the reference's path for Python callers (tests, bench.py).

The reference has no API to mirror -- only main() programs -- so the class below follows the order of
serial.c's main: load patterns (serial.c:54-87), load payloads (serial.c:91-141), build the failure
tables (serial.c:148-152), count (serial.c:153-155), report (serial.c:163-168).  All compute happens
in libkmpb200.so on the GPU; numpy/torch only carry buffers.
"""
import ctypes
import io
import os
import tempfile

import numpy as np

from . import _lib
from ._lib import CCsr, CPatterns, CSynth, KmpbError, c_i32p, c_u8p, c_u32p, c_u64p, check, lib

ENGINE_AUTO, ENGINE_PERPAT, ENGINE_UNION = 0, 1, 2
PROTO_UDP, PROTO_TCP = 0, 1
_PROTO = {"udp": PROTO_UDP, "tcp": PROTO_TCP, PROTO_UDP: PROTO_UDP, PROTO_TCP: PROTO_TCP}
FIND_SORTED = 1
# one kmpb_match record (include/kmpb200.h): where a pattern occurs
MATCH_DTYPE = np.dtype([("packet", "<u8"), ("offset", "<u4"), ("pattern", "<u4")])
_ENGINE = {"auto": ENGINE_AUTO, "perpat": ENGINE_PERPAT, "union": ENGINE_UNION,
           ENGINE_AUTO: ENGINE_AUTO, ENGINE_PERPAT: ENGINE_PERPAT, ENGINE_UNION: ENGINE_UNION}


def _as_u8(buf):
    a = np.frombuffer(buf, dtype=np.uint8) if isinstance(buf, (bytes, bytearray, memoryview)) else np.ascontiguousarray(buf, dtype=np.uint8)
    return a if a.size else np.zeros(1, dtype=np.uint8)


def pack_patterns(patterns):
    """list of bytes -> (blob uint8[], pat_off uint32[n+1]) as kmpb_set_patterns wants them."""
    patterns = [bytes(p) for p in patterns]
    blob = _as_u8(b"".join(patterns)).copy()
    off = np.zeros(len(patterns) + 1, dtype=np.uint32)
    if patterns:
        np.cumsum([len(p) for p in patterns], out=off[1:])
    return blob, off


def device_count():
    return lib().kmpb_device_count()


def shard_range(n_packets, world, rank):
    """mpi_dumping.c:149-157: (first, count) of rank's contiguous packet slice."""
    first, count = ctypes.c_uint64(0), ctypes.c_uint64(0)
    lib().kmpb_shard_range(n_packets, world, rank, ctypes.byref(first), ctypes.byref(count))
    return first.value, count.value


def extract_payload(frame, proto="udp"):
    """(offset, length) of the payload inside an Ethernet frame, or None (packet_dumping.h:87-188)."""
    f = _as_u8(frame)
    off, plen = ctypes.c_uint32(0), ctypes.c_uint32(0)
    fn = lib().kmpb_extract_tcp if _PROTO[proto] == PROTO_TCP else lib().kmpb_extract_udp
    ok = fn(f.ctypes.data_as(c_u8p), len(frame), ctypes.byref(off), ctypes.byref(plen))
    return (off.value, plen.value) if ok else None


def load_patterns(path):
    """serial.c:54-87: the whitespace-separated tokens of a strings file, in order, duplicates kept."""
    cp = CPatterns()
    check(lib().kmpb_load_patterns_file(os.fsencode(path), ctypes.byref(cp)))
    try:
        offs = [cp.pat_off[i] for i in range(cp.n_pat + 1)]
        data = ctypes.string_at(cp.blob, offs[-1]) if offs[-1] else b""
        return [data[offs[i]:offs[i + 1]] for i in range(cp.n_pat)]
    finally:
        lib().kmpb_free_patterns(ctypes.byref(cp))


class PayloadBatch:
    """Flat CSR batch of payloads produced by the C packer (serial.c:91-141).  `data` / `offsets` are
    numpy views of the C buffers (pinned when pinned=True); keep the object alive while they are used."""

    def __init__(self, path, proto="udp", pinned=False):
        self._c = CCsr()
        check(lib().kmpb_load_pcap_csr(os.fsencode(path), _PROTO[proto], 1 if pinned else 0, ctypes.byref(self._c)))
        c = self._c
        self.n_packets, self.n_frames, self.total_bytes = c.n_packets, c.n_frames, c.total_bytes
        self.offsets = np.ctypeslib.as_array(c.offsets, shape=(c.n_packets + 1,))
        self.data = np.ctypeslib.as_array(c.bytes, shape=(max(c.total_bytes, 1),))[: c.total_bytes]

    def close(self):
        if self._c is not None:
            self.data = self.offsets = None
            lib().kmpb_free_csr(ctypes.byref(self._c))
            self._c = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def format_report(patterns, counts):
    """serial.c:163-168 through the C printer: header + 'pattern: N times!' lines (bytes)."""
    blob, off = pack_patterns(patterns)
    cp = CPatterns(blob.ctypes.data_as(c_u8p), off.ctypes.data_as(c_u32p), len(patterns))
    c = np.asarray(list(counts) + [0], dtype=np.uint64)
    libc = ctypes.CDLL(None)
    libc.fopen.restype = ctypes.c_void_p
    libc.fopen.argtypes = [ctypes.c_char_p, ctypes.c_char_p]
    libc.fclose.argtypes = [ctypes.c_void_p]
    with tempfile.NamedTemporaryFile() as tmp:
        fp = libc.fopen(os.fsencode(tmp.name), b"wb")
        check(lib().kmpb_print_report(fp, ctypes.byref(cp), c.ctypes.data_as(c_u64p)))
        libc.fclose(fp)
        return open(tmp.name, "rb").read()


class Matcher:
    """One GPU context (kmpb_ctx).  Raises KmpbError(KMPB_ENODEVICE) when there is no B200: no fallback."""

    def __init__(self, device=0, engine="auto"):
        self._ctx = ctypes.c_void_p()
        check(lib().kmpb_create(ctypes.byref(self._ctx), device))
        self.device = device
        self.patterns = []
        self.set_engine(engine)

    def close(self):
        if self._ctx:
            lib().kmpb_destroy(self._ctx)
            self._ctx = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    @property
    def handle(self):
        return self._ctx

    def set_engine(self, engine):
        check(lib().kmpb_set_engine(self._ctx, _ENGINE[engine]))

    def set_patterns(self, patterns):
        """serial.c:148-152: builds the failure tables (on the device) for the whole set."""
        patterns = [bytes(p) for p in patterns]
        blob, off = pack_patterns(patterns)
        check(lib().kmpb_set_patterns(self._ctx, blob.ctypes.data_as(c_u8p), off.ctypes.data_as(c_u32p), len(patterns)))
        self.patterns = patterns

    def prefix(self, index):
        """The device-built failure table of pattern `index`, as kmp_prefix returns it (serial.c:217-238)."""
        m = len(self.patterns[index])
        out = np.zeros(m, dtype=np.int32)
        check(lib().kmpb_get_prefix(self._ctx, index, out.ctypes.data_as(c_i32p), m))
        return out.tolist()

    def count_host(self, data, offsets):
        """serial.c:153-155 over a host CSR batch -> list of per-pattern counts (file order)."""
        offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
        data = _as_u8(data)
        counts = np.zeros(max(len(self.patterns), 1), dtype=np.uint64)
        check(lib().kmpb_count_host(self._ctx, data.ctypes.data, offsets.ctypes.data, len(offsets) - 1,
                                    counts.ctypes.data_as(c_u64p)))
        return counts[: len(self.patterns)].tolist()

    def count_host_ptr(self, bytes_ptr, offsets_ptr, n_packets):
        counts = np.zeros(max(len(self.patterns), 1), dtype=np.uint64)
        check(lib().kmpb_count_host(self._ctx, bytes_ptr, offsets_ptr, n_packets, counts.ctypes.data_as(c_u64p)))
        return counts[: len(self.patterns)].tolist()

    def count_device(self, d_bytes_ptr, d_offsets_ptr, n_packets, d_counts_ptr, span=None, stream=None):
        """Asynchronous device-resident form; d_counts (uint64[n_pat]) is accumulated into."""
        if span is None:
            check(lib().kmpb_count_device(self._ctx, d_bytes_ptr, d_offsets_ptr, n_packets, d_counts_ptr, stream))
        else:
            check(lib().kmpb_count_device_span(self._ctx, d_bytes_ptr, d_offsets_ptr, n_packets, span[0], span[1],
                                               d_counts_ptr, stream))

    def count_device_into(self, d_bytes_ptr, d_offsets_ptr, n_packets, count_vector_ptrs, span, stream=None):
        """Device-resident form whose counts are added to several uint64[n_pat] vectors at once -- this GPU's
        and its peers' (NVLink-mapped) -- by the match kernel itself: count + all-reduce in one launch."""
        vecs = (ctypes.c_void_p * len(count_vector_ptrs))(*count_vector_ptrs)
        check(lib().kmpb_count_device_span_peers(self._ctx, d_bytes_ptr, d_offsets_ptr, n_packets, span[0], span[1],
                                                 vecs, len(count_vector_ptrs), stream))

    def count_pcap(self, path, proto="udp", pinned=True):
        batch = PayloadBatch(path, proto, pinned=pinned)
        try:
            return self.count_host_ptr(ctypes.cast(batch._c.bytes, ctypes.c_void_p), ctypes.cast(batch._c.offsets, ctypes.c_void_p),
                                       batch.n_packets)
        finally:
            batch.close()

    def count_pcap_streamed(self, path, proto="udp", first=0, count=None):
        """serial.c:91-155 in one pass over the savefile: batches of payloads are packed into pinned staging
        buffers and matched while the next batch is packed (kmpb_pcap_open + kmpb_count_pcap).  `first`,
        `count` select a slice of the accepted packets (a rank's share); default: all of them."""
        pc = ctypes.c_void_p()
        check(lib().kmpb_pcap_open(os.fsencode(path), _PROTO[proto], ctypes.byref(pc)))
        try:
            n = lib().kmpb_pcap_packets(pc)
            count = n - first if count is None else count
            counts = np.zeros(max(len(self.patterns), 1), dtype=np.uint64)
            check(lib().kmpb_count_pcap(self._ctx, pc, first, count, counts.ctypes.data_as(c_u64p)))
            return counts[: len(self.patterns)].tolist()
        finally:
            lib().kmpb_pcap_close(pc)

    def _find(self, call, capacity):
        """call(out_ptr, capacity, n_found_ref) once with a guessed capacity, once more with the exact total if the
        guess was short -> sorted records"""
        total = ctypes.c_uint64(0)
        for _ in range(2):
            out = np.zeros(max(capacity, 1), dtype=MATCH_DTYPE)
            check(call(out.ctypes.data, capacity, ctypes.byref(total)))
            if total.value <= capacity:
                return out[: total.value]
            capacity = total.value
        raise AssertionError("the match count changed between two runs on the same input")

    def find_host(self, data, offsets):
        """Every match in a host CSR batch (kmpb_find_host): a structured array (packet u8, offset u4, pattern u4)
        sorted by (packet, offset, pattern); pattern is the lowest index among equal patterns."""
        offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
        data = _as_u8(data)
        n = len(offsets) - 1
        guess = (int(offsets[-1]) - int(offsets[0])) // 256 + 1024 if n > 0 else 0
        return self._find(lambda out, cap, nf: lib().kmpb_find_host(self._ctx, data.ctypes.data, offsets.ctypes.data, n,
                                                                    out, cap, nf), guess)

    def find_host_ptr(self, bytes_ptr, offsets_ptr, n_packets, capacity_guess):
        """find_host over raw host pointers (bytes_ptr is absolute byte 0 of the offsets), like count_host_ptr"""
        return self._find(lambda out, cap, nf: lib().kmpb_find_host(self._ctx, bytes_ptr, offsets_ptr, n_packets, out, cap, nf),
                          capacity_guess)

    def find_pcap(self, path, proto="udp", first=0, count=None):
        """Every match in accepted packets [first, first+count) of a savefile (kmpb_find_pcap), sorted; `packet` is the
        accepted-packet index and the added field `frame` (u8) the 0-based capture record number it came from."""
        pc = ctypes.c_void_p()
        check(lib().kmpb_pcap_open(os.fsencode(path), _PROTO[proto], ctypes.byref(pc)))
        try:
            n = lib().kmpb_pcap_packets(pc)
            count = n - first if count is None else count
            guess = lib().kmpb_pcap_bytes(pc) // 256 + 1024
            rec = self._find(lambda out, cap, nf: lib().kmpb_find_pcap(self._ctx, pc, first, count, out, cap, nf), guess)
            frames = np.zeros(max(count, 1), dtype=np.uint64)
            check(lib().kmpb_pcap_frame_index(pc, first, count, frames.ctypes.data))
        finally:
            lib().kmpb_pcap_close(pc)
        out = np.zeros(len(rec), dtype=MATCH_DTYPE.descr + [("frame", "<u8")])
        for f in ("packet", "offset", "pattern"):
            out[f] = rec[f]
        out["frame"] = frames[(rec["packet"] - first).astype(np.int64)]
        return out

    def find_device(self, d_bytes, d_offsets, n_packets, d_out, capacity, d_n_found, span, sorted=False, stream=None):
        """kmpb_find_device_span: asynchronous; d_out (kmpb_match[capacity]) and d_n_found (uint64, overwritten with
        the total) are device pointers."""
        check(lib().kmpb_find_device_span(self._ctx, d_bytes, d_offsets, n_packets, span[0], span[1], d_out, capacity,
                                          d_n_found, FIND_SORTED if sorted else 0, stream))

    def stream(self, proto="udp", batch_bytes=0):
        """Frames one at a time (the live_openmp_task.c shape): returns a FrameStream."""
        return FrameStream(self, proto, batch_bytes)

    @property
    def launches(self):
        return lib().kmpb_launch_count(self._ctx)

    def set_profile(self, on=True):
        check(lib().kmpb_set_profile(self._ctx, 1 if on else 0))

    def last_kernel_ms(self):
        out = ctypes.c_double(0)
        check(lib().kmpb_last_kernel_ms(self._ctx, ctypes.byref(out)))
        return out.value

    def last_timing_ms(self):
        out = (ctypes.c_double * 2)()
        check(lib().kmpb_last_timing(self._ctx, out, 2))
        return out[0], out[1]


class FrameStream:
    """kmpb_stream_*: push captured frames; batches are matched on the GPU while pushing goes on."""

    def __init__(self, matcher, proto="udp", batch_bytes=0):
        self._m = matcher
        self._s = ctypes.c_void_p()
        check(lib().kmpb_stream_open(matcher.handle, _PROTO[proto], batch_bytes, ctypes.byref(self._s)))

    def push(self, frame):
        frame = bytes(frame)
        check(lib().kmpb_stream_push(self._s, frame, len(frame)))

    def flush(self):
        counts = np.zeros(max(len(self._m.patterns), 1), dtype=np.uint64)
        check(lib().kmpb_stream_flush(self._s, counts.ctypes.data_as(c_u64p)))
        return counts[: len(self._m.patterns)].tolist()

    @property
    def packets(self):
        return lib().kmpb_stream_packets(self._s)

    def close(self):
        if self._s:
            lib().kmpb_stream_close(self._s)
            self._s = ctypes.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


class Synth:
    """Counter-based synthetic UDP payload stream (csrc/cuda/synth.cu): BASELINE configs 3-5."""

    def __init__(self, seed=0xB200, payload_len=1400, len_mode=0, plants=2, plant_patterns=()):
        self._blob, self._off = pack_patterns(plant_patterns)
        self.cfg = CSynth(seed, payload_len, len_mode, plants if plant_patterns else 0,
                          self._blob.ctypes.data_as(c_u8p), self._off.ctypes.data_as(c_u32p), len(plant_patterns))

    def nbytes(self, first, count):
        return lib().kmpb_synth_bytes(ctypes.byref(self.cfg), first, count)

    def fill_host(self, first, count, data=None, offsets=None):
        total = self.nbytes(first, count)
        if data is None:
            data = np.zeros(total + 64, dtype=np.uint8)
        if offsets is None:
            offsets = np.zeros(count + 1, dtype=np.uint64)
        check(lib().kmpb_synth_fill_host(ctypes.byref(self.cfg), first, count, data.ctypes.data, offsets.ctypes.data))
        return data[:total], offsets

    def fill_device(self, matcher, first, count, d_bytes_ptr, d_offsets_ptr):
        check(lib().kmpb_synth_fill_device(matcher.handle, ctypes.byref(self.cfg), first, count, d_bytes_ptr, d_offsets_ptr))
