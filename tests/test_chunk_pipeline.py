"""The chunked find forms when a chunk finds more records than its stream slot's buffer holds.  That buffer starts at
about one record per 256 bytes of the plan's largest chunk; retiring a chunk that overflowed it matches the chunk again,
from the copy still on the device, into a buffer of the exact size.  A one-byte pattern over runs of that byte
overflows it many times over."""
import numpy as np
import pytest

from test_find import RefFinder, assert_invariant, csr
from test_host import _udp_frame, _write_pcap

import multithreading_string_matching_b200 as kmp


@pytest.mark.gpu
def test_find_records_past_the_slot_buffer(monkeypatch, tmp_path):
    monkeypatch.setenv("KMPB_CHUNK_MB", "1")  # 256 packets of 4096 bytes a chunk: 5 chunks, slot 0 takes two
    sparse = (b"x" * 511 + b"a") * 8  # 8 records a packet: the first chunk fits its slot's buffer
    packets = [sparse] * 256 + [b"a" * 4096] * 1024  # 4096 records a packet: every later chunk overflows it
    data, offsets = csr(packets)
    patterns = [b"a"]
    want = RefFinder(str(tmp_path)).find_csr(data, offsets, patterns)
    assert len(want) == 256 * 8 + 1024 * 4096
    path = str(tmp_path / "dense.pcap")
    _write_pcap(path, [_udp_frame(p) for p in packets])
    with kmp.Matcher(0) as m:
        m.set_patterns(patterns)
        counts = m.count_host(data, offsets)
        got = m.find_host(data, offsets)
        assert np.array_equal(got, want)
        assert_invariant(counts, got, patterns)
        got = m.find_pcap(path)[["packet", "offset", "pattern"]].astype(kmp.MATCH_DTYPE)
        assert np.array_equal(got, want)
        assert_invariant(counts, got, patterns)
