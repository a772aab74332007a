"""Where the patterns occur: kmpb_find_* (the union engine's find kernel, the locate and sort steps), Matcher.find_*,
bin/kmp_find.  The reference finder, kmpo_find_csr (tests/c/kmp_find_ref.c, a restatement of the reference's
kmp_matcher that records where it hits), is checked against a naive finder and against the oracle's counts; the CPU
tests also check the host side of the savefile frame numbers.  The GPU tests check every find form against the
reference finder's sorted records and against the count forms on the same input (for every pattern i, counts[i] = the
records carrying i's first index)."""
import ctypes
import os
import random
import subprocess

import numpy as np
import pytest

from conftest import DATA, golden_runs
from kmpb_harness import (FIND, FIND_FORMS, FIND_HOST_FORMS, PCAPS, DeviceBatch, check_forms, pcap_frames, udp_frame,
                          write_pcap)
from kmpb_reference import ORDER, as_tuples, assert_invariant, csr, finder, firsts, naive

import multithreading_string_matching_b200 as kmp


# ---- CPU ------------------------------------------------------------------------------------------

def test_reference_finder_against_a_naive_one(oracle):
    rng = random.Random(31)
    cases = [
        ([b"aaaa", b"xaax\0aa", b"", b"aa"], [b"aa", b"a", b"aa", b"aaa"]),     # overlaps, NUL cut, duplicates
        ([b"http", b"xhttp", b"htt", b"ht\0tp"], [b"http", b"t", b"p"]),     # ends at the packet's end, cut short
        ([b"x" * 150], [b"x" * 99, b"x"]),                                  # 1- and 99-byte patterns
        ([b"abc"], []),
        ([], [b"a"]),
    ]
    for _ in range(60):
        alpha = rng.choice([b"ab", b"ab\0", b"abcd", bytes(range(1, 256))])
        pats = [bytes(rng.choice(alpha.replace(b"\0", b"") or b"a") for _ in range(rng.choice([1, 1, 2, 3, 5, 9, 99])))
                for _ in range(rng.randint(1, 8))]
        pats += rng.sample(pats, min(2, len(pats)))
        pkts = [bytes(rng.choice(alpha) for _ in range(rng.choice([0, 1, 3, 17, 120, 400]))) for _ in range(rng.randint(0, 12))]
        cases.append((pkts, pats))
    for pkts, pats in cases:
        data, offsets = csr(pkts)
        got = as_tuples(finder().find_csr(data, offsets, pats))
        assert got == naive(pkts, pats), (pkts[:3], pats)
        counts = oracle.count_csr(data, offsets, pats)
        first = firsts(pats)
        assert counts == [sum(1 for r in got if r[2] == first[i]) for i in range(len(pats))]


def test_find_needs_a_device(tmp_path):
    """No CPU path: without a B200 no context exists to find with, the find entry points refuse a NULL context, and
    kmp_find stops with the message kmp_match gives."""
    import torch

    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    with pytest.raises(kmp.KmpbError) as e:
        kmp.Matcher()
    assert e.value.code == -4
    lib = kmp.lib()
    n = ctypes.c_uint64(0)
    assert lib.kmpb_find_host(None, None, None, 0, None, 0, ctypes.byref(n)) == -1
    assert lib.kmpb_find_pcap(None, None, 0, 0, None, 0, ctypes.byref(n)) == -1
    assert lib.kmpb_find_device_span(None, None, None, 0, 0, 0, None, 0, None, 0, None) == -1
    r = subprocess.run([FIND, os.path.join(DATA, "udp.pcap"), os.path.join(DATA, "strings.txt")], capture_output=True, text=True)
    assert r.returncode == 1 and "no CPU path" in r.stderr and r.stdout == ""


def test_kmp_find_usage_and_errors(tmp_path):
    r = subprocess.run([FIND], capture_output=True, text=True)
    assert r.returncode == 1 and r.stdout == "USAGE: ./kmp_find <file.pcap> <string.txt> [tcp/udp]\n"
    r = subprocess.run([FIND, "a", "b", "icmp"], capture_output=True, text=True)
    assert r.returncode == 1 and r.stdout.startswith("USAGE ")
    r = subprocess.run([FIND, os.path.join(DATA, "udp.pcap"), str(tmp_path / "missing.txt")], capture_output=True, text=True)
    assert r.returncode == 1 and r.stderr.startswith("error opening file: ")


@pytest.mark.parametrize("pcap", PCAPS)
@pytest.mark.parametrize("proto", ["udp", "tcp"])
def test_pcap_frame_index_is_the_accepted_frames(oracle, pcap, proto):
    path = os.path.join(DATA, pcap + ".pcap")
    want = [i for i, f in enumerate(pcap_frames(path)) if oracle.extract(f, proto) is not None]
    lib = kmp.lib()
    pc = ctypes.c_void_p()
    kmp.matcher.check(lib.kmpb_pcap_open(os.fsencode(path), kmp.matcher._PROTO[proto], ctypes.byref(pc)))
    try:
        n = lib.kmpb_pcap_packets(pc)
        assert n == len(want)
        frames = np.zeros(max(n, 1), dtype=np.uint64)
        kmp.matcher.check(lib.kmpb_pcap_frame_index(pc, 0, n, frames.ctypes.data))
        assert frames[:n].tolist() == want
        if n > 3:
            part = np.zeros(2, dtype=np.uint64)
            kmp.matcher.check(lib.kmpb_pcap_frame_index(pc, n - 3, 2, part.ctypes.data))
            assert part.tolist() == want[n - 3:n - 1]
        assert lib.kmpb_pcap_frame_index(pc, n, 1, frames.ctypes.data) == -1
    finally:
        lib.kmpb_pcap_close(pc)


# ---- GPU ------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def matcher():
    m = kmp.Matcher(0)
    yield m
    m.close()


@pytest.fixture(scope="module")
def strings(strings_txt):
    return kmp.load_patterns(strings_txt)


@pytest.mark.gpu
@pytest.mark.parametrize("pcap,proto,expected", golden_runs(), ids=lambda v: v if isinstance(v, str) else "")
def test_bundled_pcaps(matcher, oracle, strings, pcap, proto, expected):
    path = os.path.join(DATA, pcap + ".pcap")
    data, offsets, _ = oracle.load_pcap_csr(path, proto)
    want = finder().find_csr(data, offsets, strings)
    matcher.set_patterns(strings)
    got = matcher.find_pcap(path, proto)
    assert np.array_equal(got[["packet", "offset", "pattern"]].astype(kmp.MATCH_DTYPE), want)
    accepted = [i for i, f in enumerate(pcap_frames(path)) if oracle.extract(f, proto) is not None]
    assert got["frame"].tolist() == [accepted[k] for k in want["packet"].tolist()]
    batch = kmp.PayloadBatch(path, proto)
    assert np.array_equal(matcher.find_host(batch.data, batch.offsets), want)
    assert_invariant(matcher.count_pcap_streamed(path, proto), want, strings)
    lines = ["%d %d %s" % (accepted[k] + 1, o, strings[p].decode("latin-1")) for k, o, p in as_tuples(want)]
    r = subprocess.run([FIND, path, os.path.join(DATA, "strings.txt"), proto], capture_output=True)
    assert r.returncode == 0, r.stderr
    assert r.stdout.decode("latin-1").splitlines() == lines


@pytest.mark.gpu
def test_semantics(matcher):
    got = check_forms((matcher,), [b"aa"], *csr([b"aaaa"]), forms=FIND_FORMS)[1]
    assert as_tuples(got) == [(0, 0, 0), (0, 1, 0), (0, 2, 0)]
    got = check_forms((matcher,), [b"ab", b"b", b"ab"], *csr([b"abab\0ab", b"\0ab", b"xab", b"ab"]), forms=FIND_FORMS)[1]
    assert as_tuples(got) == [(0, 0, 0), (0, 1, 1), (0, 2, 0), (0, 3, 1), (2, 1, 0), (2, 2, 1), (3, 0, 0), (3, 1, 1)]
    # a match ending exactly at a packet's end counts; one straddling into the next packet does not
    got = check_forms((matcher,), [b"http"], *csr([b"xxhttp", b"xxxhtt", b"pxx", b"http"]), forms=FIND_FORMS)[1]
    assert as_tuples(got) == [(0, 2, 0), (3, 0, 0)]
    check_forms((matcher,), [b"a"], *csr([]), forms=FIND_FORMS)
    check_forms((matcher,), [b"a"], *csr([b"", b"", b""]), forms=FIND_FORMS)
    matcher.set_patterns([])
    assert len(matcher.find_host(*csr([b"abc"]))) == 0


@pytest.mark.gpu
def test_pattern_lengths_1_to_99(matcher):
    rng = random.Random(99)
    pats = [bytes(rng.choice(b"abc") for _ in range(m)) for m in range(1, 100)]
    pkts = []
    for p in pats:
        for lead in (0, 1, 7, 31, 32, 33):
            pkts.append(b"c" * lead + p + b"c" * (lead % 3))
    pkts.append(b"abcabc" * 500)
    check_forms((matcher,), pats, *csr(pkts), label="lengths", forms=FIND_FORMS)


@pytest.mark.gpu
def test_random_batches(matcher):
    rng = random.Random(20261020)
    for trial in range(24):
        alpha = [b"ab", b"abc\0", bytes(range(0x20, 0x7F)), bytes(range(256))][trial % 4]
        pat_alpha = bytes(b for b in alpha if b)
        pats = [bytes(rng.choice(pat_alpha) for _ in range(rng.choice([1, 2, 3, 4, 6, 9, 20])))
                for _ in range(rng.choice([1, 3, 8, 40]))]
        equal = trial % 2 == 0  # equal-sized packets: the resolve step finds the packet by a division
        size = rng.choice([1, 33, 64, 700, 1400])
        pkts = []
        for _ in range(rng.choice([1, 10, 300, 2000])):
            n = size if equal else rng.choice([0, 1, 5, 31, 32, 33, 511, 1400, 9000])
            body = bytearray(rng.choice(alpha) for _ in range(n))
            for _ in range(rng.randint(0, 3)):
                p = rng.choice(pats)
                if len(p) <= n:
                    at = rng.randrange(0, n - len(p) + 1)
                    body[at:at + len(p)] = p
            pkts.append(bytes(body))
        check_forms((matcher,), pats, *csr(pkts), label="trial%d" % trial,
                    forms=FIND_FORMS if trial % 3 == 0 else FIND_HOST_FORMS)


@pytest.mark.gpu
def test_tiny_packets_item_edges_and_nul_dense(matcher):
    rng = random.Random(5)
    pats = [b"id", b"ack", b"http", b"content-list", b"NOTIFY", b"rr", b"a"]
    pkts = [bytes(rng.choice(b"idackhtpNOTIFYr-_cnsl \0") for _ in range(rng.choice([0, 1, 5, 16, 33, 64, 100, 200])))
            for _ in range(9000)]
    check_forms((matcher,), pats, *csr(pkts), label="tiny", forms=FIND_FORMS)
    big = [bytes(rng.choice(b"idackhtp") for _ in range(300_000)) for _ in range(2)]  # packets larger than a work item
    check_forms((matcher,), pats, *csr(big + pkts[:50]), label="big", forms=FIND_HOST_FORMS)
    for p_nul in (1.0, 0.9, 0.3):
        pkts = [bytes(0 if rng.random() < p_nul else rng.choice(b"idackhtpNOTIFY") for _ in range(rng.randint(0, 2000)))
                for _ in range(60)]
        check_forms((matcher,), pats, *csr(pkts), label="p_nul=%g" % p_nul, forms=FIND_HOST_FORMS)


@pytest.mark.gpu
def test_tables_in_global_memory(matcher):
    """700 patterns: the probe tables (and the find kernel's verification) run from global memory."""
    rng = random.Random(4242)
    alpha = b"abcdefgh01"
    pats = [bytes(rng.choice(alpha) for _ in range(rng.choice([1, 2, 3, 4, 8, 9, 13, 41, 99]))) for _ in range(700)]
    pats += pats[:20]
    pkts = []
    for _ in range(300):
        body = bytearray(rng.choice(alpha) for _ in range(rng.choice([0, 40, 700, 3000])))
        for _ in range(rng.randint(0, 4)):
            p = rng.choice(pats)
            if len(p) <= len(body):
                at = rng.randrange(0, len(body) - len(p) + 1)
                body[at:at + len(p)] = p
        pkts.append(bytes(body))
    check_forms((matcher,), pats, *csr(pkts), label="720 patterns", forms=FIND_FORMS)


@pytest.mark.gpu
def test_device_form_capacity(matcher, strings):
    synth = kmp.Synth(seed=0xB200, payload_len=1400, plants=2, plant_patterns=strings)
    data, offsets = synth.fill_host(0, 5000)
    matcher.set_patterns(strings)
    want = finder().find_csr(data, offsets, strings)
    total = len(want)
    assert total > 1000
    wanted = set(as_tuples(want))
    batch = DeviceBatch(data, offsets)
    for cap in (0, 1, total // 3, total - 1):
        for sorted_ in (False, True):
            rec, n, ok = batch.find(matcher, cap, sorted_)
            got = as_tuples(rec)
            assert n == total and ok and len(got) == cap and len(set(got)) == cap and set(got) <= wanted, (cap, sorted_)
    rec, n, ok = batch.find(matcher, total, True)
    assert n == total and ok and np.array_equal(rec, want)
    rec, n, ok = batch.find(matcher, total + 100, False)
    assert n == total and ok and np.array_equal(np.sort(rec, order=ORDER), want)
    # the host forms with a short buffer: the first records in sorted order, the exact total
    out = np.zeros(100, dtype=kmp.MATCH_DTYPE)
    n = ctypes.c_uint64(0)
    kmp.matcher.check(kmp.lib().kmpb_find_host(matcher.handle, data.ctypes.data, offsets.ctypes.data, len(offsets) - 1,
                                               out.ctypes.data, 100, ctypes.byref(n)))
    assert n.value == total and np.array_equal(out, want[:100])
    assert kmp.lib().kmpb_find_device_span(matcher.handle, None, None, 0, 0, 0, None, 0, out.ctypes.data, 2, None) == -1


@pytest.mark.gpu
def test_many_chunks_and_slices(matcher, oracle, strings, monkeypatch, tmp_path):
    monkeypatch.setenv("KMPB_CHUNK_MB", "1")
    synth = kmp.Synth(seed=7, len_mode=1, plants=2, plant_patterns=strings)
    data, offsets = synth.fill_host(0, 12000)  # ~20 MB of mixed sizes: ~20 chunks, every slot reused
    matcher.set_patterns(strings)
    want = finder().find_csr(data, offsets, strings)
    assert np.array_equal(matcher.find_host(data, offsets), want)
    path = os.path.join(DATA, "very_big_udp.pcap")
    pdata, poffsets, _ = oracle.load_pcap_csr(path, "udp")
    pwant = finder().find_csr(pdata, poffsets, strings)
    n = len(poffsets) - 1
    assert np.array_equal(matcher.find_pcap(path)[["packet", "offset", "pattern"]].astype(kmp.MATCH_DTYPE), pwant)
    for first, count in ((0, 1), (100, 5000), (n - 7000, 7000), (n, 0)):
        got = matcher.find_pcap(path, first=first, count=count)
        sel = pwant[(pwant["packet"] >= first) & (pwant["packet"] < first + count)]
        assert np.array_equal(got[["packet", "offset", "pattern"]].astype(kmp.MATCH_DTYPE), sel), (first, count)
    # Plans of exactly 1, KMPB_COPY_STREAMS (4) and KMPB_COPY_STREAMS + 1 chunks (a 1 MiB chunk is 256 packets of 4096
    # bytes), and a packet of over 3 MiB, larger than a chunk: the four host and savefile forms against the oracle and
    # the reference finder
    sdata, soff = kmp.Synth(seed=11, payload_len=4096, plants=2, plant_patterns=strings).fill_host(0, 5 * 256)
    pkts = [bytes(sdata[int(a):int(b)]) for a, b in zip(soff[:-1], soff[1:])]
    assert {len(p) for p in pkts} == {4096}
    rng = np.random.default_rng(11)
    giant = bytearray(rng.choice(np.frombuffer(b"acdeikoprstu ", np.uint8), (3 << 20) + 123).tobytes())
    for at in rng.integers(0, len(giant) - 16, 500).tolist():
        p = strings[at % len(strings)]
        giant[at:at + len(p)] = p
    for label, case in (("1 chunk", pkts[:256]), ("4 chunks", pkts[:1024]), ("5 chunks", pkts),
                        ("a packet larger than a chunk", pkts[:300] + [bytes(giant)] + pkts[300:600])):
        data, offsets = csr(case)
        path = str(tmp_path / "chunks.pcap")
        write_pcap(path, [udp_frame(p) for p in case])
        counts = oracle.count_csr(data, offsets, strings)
        want = finder().find_csr(data, offsets, strings)
        assert len(want) > 1000, label
        assert matcher.count_host(data, offsets) == counts, label
        assert matcher.count_pcap_streamed(path) == counts, label
        got = matcher.find_host(data, offsets)
        assert np.array_equal(got, want), label
        assert_invariant(counts, got, strings)
        got = matcher.find_pcap(path)[["packet", "offset", "pattern"]].astype(kmp.MATCH_DTYPE)
        assert np.array_equal(got, want), label
        assert_invariant(counts, got, strings)


@pytest.mark.gpu
def test_count_before_and_after_find(matcher, oracle, strings):
    synth = kmp.Synth(seed=0xB200, payload_len=1400, plants=2, plant_patterns=strings)
    data, offsets = synth.fill_host(0, 3000)
    matcher.set_patterns(strings)
    batch = DeviceBatch(data, offsets)

    def counts():
        return matcher.count_host(data, offsets), batch.count(matcher)[0]

    before = counts()
    rec = matcher.find_host(data, offsets)
    batch.find(matcher, 10, True)
    assert counts() == before
    assert before[0] == before[1] == oracle.count_csr(data, offsets, strings)
    assert_invariant(before[0], rec, strings)
    matcher.set_engine("perpat")  # finding runs the union engine whatever the engine setting
    try:
        assert np.array_equal(matcher.find_host(data, offsets), rec)
    finally:
        matcher.set_engine("auto")
