"""How inputs are built and forms are driven: the binaries, hand-built savefiles, a batch on the device with the device
forms run on it, the two engines, and one check of any set of forms against the expected answers
(tests/kmpb_reference.py)."""
import ctypes
import os
import struct
import subprocess

import numpy as np
import pytest

from conftest import DATA, ROOT
from kmpb_reference import ORDER, as_tuples, expected, normalise

import multithreading_string_matching_b200 as kmp

BIN = os.path.join(ROOT, "multithreading_string_matching_b200", "bin")
MATCH, FIND, SELECT = (os.path.join(BIN, b) for b in ("kmp_match", "kmp_find", "kmp_select"))
STRINGS = os.path.join(DATA, "strings.txt")
PCAPS = ["udp", "udp_1000", "big_udp", "very_big_udp", "tcp"]


# ---- savefiles ------------------------------------------------------------------------------------------------------

def udp_frame(payload, proto=17, ihl=5):
    """Ethernet + IPv4 (ihl words) + UDP header + payload"""
    ip = bytes([0x40 | ihl, 0, 0, 0, 0, 0, 0, 0, 64, proto]) + b"\0" * (ihl * 4 - 10)
    return b"\x02" * 12 + b"\x08\x00" + ip + b"\0" * 8 + bytes(payload)


def write_pcap(path, frames, magic=0xA1B2C3D4, swapped=False, caplens=None):
    e = ">" if swapped else "<"
    with open(path, "wb") as f:
        f.write(struct.pack(e + "IHHiIII", magic, 2, 4, 0, 0, 262144, 1))
        for i, fr in enumerate(frames):
            cap = len(fr) if caplens is None else caplens[i]
            f.write(struct.pack(e + "IIII", 1, 2, cap, len(fr)))
            f.write(fr[:cap])


def pcapng(frames, big_endian=False, simple_from=None, second_section_at=None, packet_blocks=False):
    """A pcapng file by hand: SHB, IDB, one packet block per frame (Enhanced; Simple from index `simple_from` on;
    obsolete Packet Blocks and an Interface Statistics Block at the end with `packet_blocks`), a name-resolution block
    in the middle, optionally a second section in the other byte order."""

    def blocks(frames, e, first_index):
        def block(btype, body):
            body += b"\0" * (-len(body) % 4)
            total = len(body) + 12
            return struct.pack(e + "II", btype, total) + body + struct.pack(e + "I", total)

        out = block(0x0A0D0D0A, struct.pack(e + "IHHq", 0x1A2B3C4D, 1, 0, -1) + struct.pack(e + "HH", 2, 5) + b"shark\0\0\0" + struct.pack(e + "HH", 0, 0))
        out += block(1, struct.pack(e + "HHI", 1, 0, 262144))
        for k, f in enumerate(frames):
            if k == 1:
                out += block(4, b"\0" * 8)  # a Name Resolution Block: skipped
            if packet_blocks:
                out += block(2, struct.pack(e + "HHIIII", 0, 0, 0, k, len(f), len(f)) + f)
            elif simple_from is not None and first_index + k >= simple_from:
                out += block(3, struct.pack(e + "I", len(f)) + f)
            else:
                out += block(6, struct.pack(e + "IIIII", 0, 0, k, len(f), len(f)) + f + b"\0" * (-len(f) % 4) + struct.pack(e + "HHI", 1, 4, 0x64636261) + struct.pack(e + "HH", 0, 0))
        if packet_blocks:
            out += block(5, struct.pack(e + "III", 0, 0, 0))
        return out

    e = ">" if big_endian else "<"
    if second_section_at is None:
        return blocks(frames, e, 0)
    other = "<" if big_endian else ">"
    return blocks(frames[:second_section_at], e, 0) + blocks(frames[second_section_at:], other, second_section_at)


def classic_records(path):
    """(global header, [whole record bytes]) of a classic savefile, up to a cut trailing record"""
    raw = open(path, "rb").read()
    e = "<" if struct.unpack("<I", raw[:4])[0] in (0xA1B2C3D4, 0xA1B23C4D) else ">"
    at, recs = 24, []
    while len(raw) - at >= 16:
        cap = struct.unpack(e + "I", raw[at + 8:at + 12])[0]
        if cap > len(raw) - at - 16:
            break
        recs.append(raw[at:at + 16 + cap])
        at += 16 + cap
    return raw[:24], recs


def pcap_frames(path):
    """the captured bytes of every record of a classic savefile, in file order"""
    return [r[16:] for r in classic_records(path)[1]]


def build_integration_snippet(tmp_path):
    """tests/c/integration_snippet.c (the call sequence of INTEGRATION.md section 1) against include/kmpb200.h and
    libkmpb200.so only."""
    exe = str(tmp_path / "integration_snippet")
    pkg = os.path.join(ROOT, "multithreading_string_matching_b200")
    subprocess.run(["/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc", "-O1", "-g", "-Wall", "-Wextra", "-Werror",
                    "-I" + os.path.join(ROOT, "include"), os.path.join(ROOT, "tests", "c", "integration_snippet.c"),
                    "-L" + pkg, "-lkmpb200", "-Wl,-rpath," + pkg, "-o", exe], check=True)
    return exe


# ---- the device forms -----------------------------------------------------------------------------------------------

class DeviceBatch:
    """A CSR batch on cuda:0 and the device forms run on packets [k0, k1) of it, each waited for.  Their outputs start
    non-zero -- counts at 3 (select: 5), find buffers 0xA5 behind the capacity -- so that a form that overwrites
    instead of adding, or writes past the capacity, shows."""

    def __init__(self, data, offsets):
        """a copy of the batch: its bytes (a multiple of 32, at least 64 bytes of zeros behind the data), its offsets"""
        import torch

        self.d_bytes = torch.zeros(((len(data) + 64 + 31) // 32) * 32, dtype=torch.uint8, device="cuda:0")
        if len(data):
            self.d_bytes[: len(data)] = torch.from_numpy(np.array(data, dtype=np.uint8)).cuda()
        self.d_off = torch.from_numpy(np.ascontiguousarray(offsets, dtype=np.int64)).cuda()
        self.offsets = np.asarray(offsets)

    @classmethod
    def on_device(cls, d_bytes, d_off, offsets):
        """a batch already on the device; `offsets` is the host copy of d_off"""
        b = cls.__new__(cls)
        b.d_bytes, b.d_off, b.offsets = d_bytes, d_off, np.asarray(offsets)
        return b

    def _args(self, k0, k1):
        k1 = len(self.offsets) - 1 if k1 is None else k1
        return (self.d_bytes.data_ptr(), self.d_off.data_ptr() + 8 * k0, k1 - k0), (int(self.offsets[k0]), int(self.offsets[k1]))

    def count(self, m, n_vectors=1, k0=0, k1=None):
        """kmpb_count_device_span (n_vectors = 1) or _span_peers into n_vectors vectors -> the vectors"""
        import torch

        batch, span = self._args(k0, k1)
        vecs = [torch.full((max(len(m.patterns), 1),), 3, dtype=torch.int64, device="cuda:0") for _ in range(n_vectors)]
        if n_vectors == 1:
            m.count_device(*batch, vecs[0].data_ptr(), span=span)
        else:
            m.count_device_into(*batch, [v.data_ptr() for v in vecs], span)
        torch.cuda.synchronize()
        return [[c - 3 for c in v[: len(m.patterns)].cpu().tolist()] for v in vecs]

    def find(self, m, capacity, sorted_=True, k0=0, k1=None, canary=8):
        """kmpb_find_device_span -> (records written, total, canary intact)"""
        import torch

        batch, span = self._args(k0, k1)
        d_out = torch.full(((capacity + canary) * 16,), 0xA5, dtype=torch.uint8, device="cuda:0")
        d_n = torch.full((1,), -1, dtype=torch.int64, device="cuda:0")
        m.find_device(*batch, d_out.data_ptr(), capacity, d_n.data_ptr(), span, sorted=sorted_)
        torch.cuda.synchronize()
        total = int(d_n.item())
        rec = d_out[: 16 * min(total, capacity)].cpu().numpy().view(kmp.MATCH_DTYPE)
        return rec, total, bool((d_out[16 * capacity:] == 0xA5).all().item())

    def select(self, m, k0=0, k1=None, invert=False, stream=None, wait=True):
        """kmpb_select_device_span -> (flags, index list, counts); with wait=False, on `stream`, a function that reads
        them once the caller has waited"""
        import torch

        batch, span = self._args(k0, k1)
        n, n_pat = batch[2], len(m.patterns)
        d_flags = torch.full((max(n, 1),), 7, dtype=torch.uint8, device="cuda:0")
        d_index = torch.full((max(n, 1),), -1, dtype=torch.int64, device="cuda:0")
        d_n = torch.full((1,), -1, dtype=torch.int64, device="cuda:0")
        d_counts = torch.full((max(n_pat, 1),), 5, dtype=torch.int64, device="cuda:0")
        m.select_device(*batch, d_flags.data_ptr(), span, d_index.data_ptr(), d_n.data_ptr(), d_counts.data_ptr(),
                        invert=invert, stream=stream)

        def results():
            return (d_flags[:n].cpu().numpy().astype(bool), d_index[: int(d_n.item())].cpu().numpy(),
                    [c - 5 for c in d_counts[:n_pat].cpu().tolist()])

        if wait:
            torch.cuda.synchronize()
            return results()
        return results


@pytest.fixture(scope="module")
def engines():
    """(union, per-pattern) contexts of one test module"""
    u, p = kmp.Matcher(0, engine="union"), kmp.Matcher(0, engine="perpat")
    yield u, p
    u.close()
    p.close()


HOST_FORMS = ("count_host", "find_host", "select_host")
DEVICE_FORMS = ("count_device", "find_device", "find_short", "select_device")
FIND_HOST_FORMS = ("count_host", "find_host")
FIND_FORMS = FIND_HOST_FORMS + ("find_device",)
SELECT_FORMS = ("count_host", "select_host", "select_bare", "select_device", "select_inverted")


def check_forms(engines, patterns, data, offsets, nocase=False, window=None, forms=HOST_FORMS + DEVICE_FORMS, label="",
                answers=None, oracle=None):
    """Sets the patterns on every engine and checks `forms` against `answers` (counts, sorted records, verdicts), by
    default kmpb_reference.expected's; returns them.  The count forms run on every engine, the others on the first.
      count_host     kmpb_count_host
      find_host      kmpb_find_host
      select_host    kmpb_select_host: verdicts and counts
      select_bare    kmpb_select_host without counts_out: verdicts and the number selected
      count_device   kmpb_count_device_span into one vector and _span_peers into three
      find_device    kmpb_find_device_span, sorted and unsorted, capacity = the number of records (batches of packets)
      find_short     unsorted, one record short: the exact total, a subset written (batches with records)
      select_device  kmpb_select_device_span: verdicts, index list, counts
      select_inverted  the same with invert"""
    counts, rec, verdicts = answers if answers is not None else expected(patterns, data, offsets, nocase, window, oracle)
    first = engines[0]
    for m in engines:
        m.set_patterns(patterns, nocase, window)
    assert first.nocase == normalise(patterns, nocase)[1]
    n = len(offsets) - 1
    if "count_host" in forms:
        for m in engines:
            assert m.count_host(data, offsets) == counts, (label, "count_host", m is first)
    if "find_host" in forms:
        got = first.find_host(data, offsets)
        assert got.dtype == kmp.MATCH_DTYPE
        if not np.array_equal(got, rec):
            w, g = set(as_tuples(rec)), set(as_tuples(got))
            raise AssertionError((label, len(rec), len(got), sorted(w - g)[:5], sorted(g - w)[:5]))
    if "select_host" in forms:
        flags, c = first.select_host(data, offsets)
        assert np.array_equal(flags, verdicts), (label, "select_host", np.flatnonzero(flags != verdicts)[:8])
        assert c == counts, (label, "select_host counts")
    if "select_bare" in forms:
        d = np.array(data, dtype=np.uint8) if len(data) else np.zeros(1, np.uint8)
        o = np.ascontiguousarray(offsets, dtype=np.uint64)
        fl = np.zeros(max(n, 1), dtype=np.uint8)
        n_sel = ctypes.c_uint64(12345)
        kmp.matcher.check(kmp.lib().kmpb_select_host(first.handle, d.ctypes.data, o.ctypes.data, n, fl.ctypes.data,
                                                     ctypes.byref(n_sel), None))
        assert n_sel.value == int(verdicts.sum()) and np.array_equal(fl[:n].astype(bool), verdicts), (label, "select_bare")
    if not any(f in DEVICE_FORMS + ("select_inverted",) for f in forms):
        return counts, rec, verdicts
    batch = DeviceBatch(data, offsets)
    if "count_device" in forms:
        for m in engines:
            assert batch.count(m) == [counts], (label, "count_device", m is first)
            assert batch.count(m, 3) == [counts] * 3, (label, "count_device peers", m is first)
    if "find_device" in forms and n:
        got, total, ok = batch.find(first, len(rec), True)
        assert total == len(rec) and ok and np.array_equal(got, rec), (label, "find sorted")
        got, total, ok = batch.find(first, len(rec), False)
        assert total == len(rec) and ok and np.array_equal(np.sort(got, order=ORDER), rec), (label, "find unsorted")
    if "find_short" in forms and len(rec):
        got, total, ok = batch.find(first, len(rec) - 1, False)
        assert total == len(rec) and ok and len(got) == len(rec) - 1, (label, "find one short")
        assert set(as_tuples(got)) <= set(as_tuples(rec)), (label, "find one short")
    for form, invert in (("select_device", False), ("select_inverted", True)):
        if form not in forms:
            continue
        f, idx, c = batch.select(first, invert=invert)
        assert np.array_equal(f, verdicts), (label, "select_device", invert, np.flatnonzero(f != verdicts)[:8])
        assert np.array_equal(idx, np.flatnonzero(verdicts != invert)) and c == counts, (label, "select_device", invert)
    kmp.matcher.check(kmp.lib().kmpb_check_device_errors(first.handle))
    return counts, rec, verdicts
