"""Where the patterns occur: kmpb_find_* (the union engine's find kernel, the locate and sort steps), Matcher.find_*,
bin/kmp_find.  The reference finder, kmpo_find_csr (tests/c/kmp_find_ref.c, a restatement of the reference's
kmp_matcher that records where it hits), is checked against a naive finder and against the oracle's counts; the CPU
tests also check the host side of the savefile frame numbers.  The GPU tests check every find form against the
reference finder's sorted records and against the count forms on the same input (for every pattern i, counts[i] = the
records carrying i's first index)."""
import ctypes
import os
import random
import struct
import subprocess

import numpy as np
import pytest

from conftest import DATA, ROOT, golden_runs

import multithreading_string_matching_b200 as kmp

FIND = os.path.join(ROOT, "multithreading_string_matching_b200", "bin", "kmp_find")
PCAPS = ["udp", "udp_1000", "big_udp", "very_big_udp", "tcp"]


def csr(packets):
    offsets = np.zeros(len(packets) + 1, dtype=np.uint64)
    if packets:
        np.cumsum([len(p) for p in packets], out=offsets[1:])
    return np.frombuffer(b"".join(packets) + b"\0" * 16, dtype=np.uint8)[: int(offsets[-1])], offsets


def first_index(patterns):
    """file-order index -> lowest index of an equal pattern"""
    seen = {}
    return [seen.setdefault(bytes(p), i) for i, p in enumerate(patterns)]


def naive_find(packets, patterns):
    firsts = first_index(patterns)
    out = []
    for k, payload in enumerate(packets):
        text = payload.split(b"\0", 1)[0]
        for i, p in enumerate(patterns):
            if firsts[i] != i:
                continue
            out += [(k, s, i) for s in range(len(text) - len(p) + 1) if text[s:s + len(p)] == p]
    return sorted(out)


def as_tuples(rec):
    return list(zip(rec["packet"].tolist(), rec["offset"].tolist(), rec["pattern"].tolist()))


def pcap_frames(path):
    """the captured bytes of every record of a classic savefile, in file order"""
    raw = open(path, "rb").read()
    e = "<" if struct.unpack("<I", raw[:4])[0] in (0xA1B2C3D4, 0xA1B23C4D) else ">"
    at, frames = 24, []
    while len(raw) - at >= 16:
        cap = struct.unpack(e + "I", raw[at + 8:at + 12])[0]
        at += 16
        if cap > len(raw) - at:
            break
        frames.append(raw[at:at + cap])
        at += cap
    return frames


class RefFinder:
    """ctypes view of tests/c/kmp_find_ref.c, compiled into `workdir`"""

    def __init__(self, workdir):
        so = os.path.join(workdir, "libkmp_find_ref.so")
        cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"
        subprocess.run([cc, "-O2", "-Wall", "-Wextra", "-Werror", "-fPIC", "-shared", "-o", so,
                        os.path.join(ROOT, "tests", "c", "kmp_find_ref.c")], check=True)
        self.lib = ctypes.CDLL(so)
        u8p, u32p, u64p = (ctypes.POINTER(t) for t in (ctypes.c_uint8, ctypes.c_uint32, ctypes.c_uint64))
        self.lib.kmpo_find_csr.restype = ctypes.c_int64
        self.lib.kmpo_find_csr.argtypes = [u8p, u64p, ctypes.c_uint64, u8p, u32p, ctypes.c_uint32, u64p, u32p, u32p,
                                           ctypes.c_int64]

    def find_csr(self, data, offsets, patterns):
        """every match of the oracle's count_csr as a record (packet, offset, lowest index of equal patterns), sorted"""
        data = np.ascontiguousarray(data, dtype=np.uint8)
        if data.size == 0:
            data = np.zeros(1, dtype=np.uint8)
        offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
        blob, off = kmp.pack_patterns(patterns)

        def p(a, t):
            return a.ctypes.data_as(ctypes.POINTER(t))

        args = (p(data, ctypes.c_uint8), p(offsets, ctypes.c_uint64), len(offsets) - 1, p(blob, ctypes.c_uint8),
                p(off, ctypes.c_uint32), len(patterns))
        total = self.lib.kmpo_find_csr(*args, None, None, None, 0)
        pk = np.zeros(max(total, 1), dtype=np.uint64)
        of = np.zeros(max(total, 1), dtype=np.uint32)
        pt = np.zeros(max(total, 1), dtype=np.uint32)
        assert self.lib.kmpo_find_csr(*args, p(pk, ctypes.c_uint64), p(of, ctypes.c_uint32), p(pt, ctypes.c_uint32), total) == total
        out = np.zeros(total, dtype=kmp.MATCH_DTYPE)
        out["packet"], out["offset"], out["pattern"] = pk[:total], of[:total], pt[:total]
        return out


@pytest.fixture(scope="module")
def finder(tmp_path_factory):
    return RefFinder(str(tmp_path_factory.mktemp("kmp_find_ref")))


# ---- CPU ------------------------------------------------------------------------------------------

def test_reference_finder_against_a_naive_one(oracle, finder):
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
        got = as_tuples(finder.find_csr(data, offsets, pats))
        assert got == naive_find(pkts, pats), (pkts[:3], pats)
        counts = oracle.count_csr(data, offsets, pats)
        firsts = first_index(pats)
        assert counts == [sum(1 for r in got if r[2] == firsts[i]) for i in range(len(pats))]


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


def assert_invariant(counts, rec, patterns):
    firsts = first_index(patterns)
    hist = np.bincount(rec["pattern"].astype(np.int64), minlength=max(len(patterns), 1))
    assert [int(hist[firsts[i]]) for i in range(len(patterns))] == list(counts)


def device_find(m, data, offsets, capacity, sorted_, canary=8):
    """kmpb_find_device_span on a device copy of the batch -> (records written, total, canary intact)"""
    import torch

    d_bytes = torch.zeros(len(data) + 64, dtype=torch.uint8, device="cuda:0")
    if len(data):
        d_bytes[: len(data)] = torch.from_numpy(np.array(data))
    d_off = torch.from_numpy(offsets.astype(np.int64)).to("cuda:0")
    d_out = torch.full(((capacity + canary) * 16,), 0xA5, dtype=torch.uint8, device="cuda:0")
    d_n = torch.full((1,), -1, dtype=torch.int64, device="cuda:0")
    span = (int(offsets[0]), int(offsets[-1])) if len(offsets) else (0, 0)
    m.find_device(d_bytes.data_ptr(), d_off.data_ptr(), len(offsets) - 1, d_out.data_ptr(), capacity, d_n.data_ptr(), span,
                  sorted=sorted_)
    torch.cuda.synchronize()
    raw = d_out.cpu().numpy()
    total = int(d_n.item())
    rec = raw[: 16 * min(total, capacity)].view(kmp.MATCH_DTYPE)
    return rec, total, bool((raw[16 * capacity:] == 0xA5).all())


def check_find(m, finder, patterns, packets, device=True, label=""):
    data, offsets = csr(packets)
    m.set_patterns(patterns)
    want = finder.find_csr(data, offsets, patterns)
    got = m.find_host(data, offsets)
    assert got.dtype == kmp.MATCH_DTYPE
    if not np.array_equal(got, want):
        w, g = set(as_tuples(want)), set(as_tuples(got))
        raise AssertionError((label, len(want), len(got), sorted(w - g)[:5], sorted(g - w)[:5]))
    assert_invariant(m.count_host(data, offsets), got, patterns)
    if device and len(packets):
        rec, total, ok = device_find(m, data, offsets, len(want), True)
        assert total == len(want) and ok and np.array_equal(rec, want), label
        rec, total, ok = device_find(m, data, offsets, len(want), False)
        assert total == len(want) and ok and np.array_equal(np.sort(rec, order=["packet", "offset", "pattern"]), want), label
    return want


@pytest.mark.gpu
@pytest.mark.parametrize("pcap,proto,expected", golden_runs(), ids=lambda v: v if isinstance(v, str) else "")
def test_bundled_pcaps(matcher, oracle, strings, pcap, proto, expected, finder):
    path = os.path.join(DATA, pcap + ".pcap")
    data, offsets, _ = oracle.load_pcap_csr(path, proto)
    want = finder.find_csr(data, offsets, strings)
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
def test_semantics(matcher, finder):
    got = check_find(matcher, finder, [b"aa"], [b"aaaa"])
    assert as_tuples(got) == [(0, 0, 0), (0, 1, 0), (0, 2, 0)]
    got = check_find(matcher, finder, [b"ab", b"b", b"ab"], [b"abab\0ab", b"\0ab", b"xab", b"ab"])
    assert as_tuples(got) == [(0, 0, 0), (0, 1, 1), (0, 2, 0), (0, 3, 1), (2, 1, 0), (2, 2, 1), (3, 0, 0), (3, 1, 1)]
    # a match ending exactly at a packet's end counts; one straddling into the next packet does not
    got = check_find(matcher, finder, [b"http"], [b"xxhttp", b"xxxhtt", b"pxx", b"http"])
    assert as_tuples(got) == [(0, 2, 0), (3, 0, 0)]
    check_find(matcher, finder, [b"a"], [])
    check_find(matcher, finder, [b"a"], [b"", b"", b""])
    matcher.set_patterns([])
    assert len(matcher.find_host(*csr([b"abc"]))) == 0


@pytest.mark.gpu
def test_pattern_lengths_1_to_99(matcher, finder):
    rng = random.Random(99)
    pats = [bytes(rng.choice(b"abc") for _ in range(m)) for m in range(1, 100)]
    pkts = []
    for p in pats:
        for lead in (0, 1, 7, 31, 32, 33):
            pkts.append(b"c" * lead + p + b"c" * (lead % 3))
    pkts.append(b"abcabc" * 500)
    check_find(matcher, finder, pats, pkts, label="lengths")


@pytest.mark.gpu
def test_random_batches(matcher, finder):
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
        check_find(matcher, finder, pats, pkts, device=trial % 3 == 0, label="trial%d" % trial)


@pytest.mark.gpu
def test_tiny_packets_item_edges_and_nul_dense(matcher, finder):
    rng = random.Random(5)
    pats = [b"id", b"ack", b"http", b"content-list", b"NOTIFY", b"rr", b"a"]
    pkts = [bytes(rng.choice(b"idackhtpNOTIFYr-_cnsl \0") for _ in range(rng.choice([0, 1, 5, 16, 33, 64, 100, 200])))
            for _ in range(9000)]
    check_find(matcher, finder, pats, pkts, label="tiny")
    big = [bytes(rng.choice(b"idackhtp") for _ in range(300_000)) for _ in range(2)]  # packets larger than a work item
    check_find(matcher, finder, pats, big + pkts[:50], device=False, label="big")
    for p_nul in (1.0, 0.9, 0.3):
        pkts = [bytes(0 if rng.random() < p_nul else rng.choice(b"idackhtpNOTIFY") for _ in range(rng.randint(0, 2000)))
                for _ in range(60)]
        check_find(matcher, finder, pats, pkts, device=False, label="p_nul=%g" % p_nul)


@pytest.mark.gpu
def test_tables_in_global_memory(matcher, finder):
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
    check_find(matcher, finder, pats, pkts, label="720 patterns")


@pytest.mark.gpu
def test_device_form_capacity(matcher, strings, finder):
    synth = kmp.Synth(seed=0xB200, payload_len=1400, plants=2, plant_patterns=strings)
    data, offsets = synth.fill_host(0, 5000)
    matcher.set_patterns(strings)
    want = finder.find_csr(data, offsets, strings)
    total = len(want)
    assert total > 1000
    wanted = set(as_tuples(want))
    for cap in (0, 1, total // 3, total - 1):
        for sorted_ in (False, True):
            rec, n, ok = device_find(matcher, data, offsets, cap, sorted_)
            got = as_tuples(rec)
            assert n == total and ok and len(got) == cap and len(set(got)) == cap and set(got) <= wanted, (cap, sorted_)
    rec, n, ok = device_find(matcher, data, offsets, total, True)
    assert n == total and ok and np.array_equal(rec, want)
    rec, n, ok = device_find(matcher, data, offsets, total + 100, False)
    assert n == total and ok and np.array_equal(np.sort(rec, order=["packet", "offset", "pattern"]), want)
    # the host forms with a short buffer: the first records in sorted order, the exact total
    out = np.zeros(100, dtype=kmp.MATCH_DTYPE)
    n = ctypes.c_uint64(0)
    kmp.matcher.check(kmp.lib().kmpb_find_host(matcher.handle, data.ctypes.data, offsets.ctypes.data, len(offsets) - 1,
                                               out.ctypes.data, 100, ctypes.byref(n)))
    assert n.value == total and np.array_equal(out, want[:100])
    assert kmp.lib().kmpb_find_device_span(matcher.handle, None, None, 0, 0, 0, None, 0, out.ctypes.data, 2, None) == -1


@pytest.mark.gpu
def test_many_chunks_and_slices(matcher, oracle, strings, monkeypatch, finder, tmp_path):
    monkeypatch.setenv("KMPB_CHUNK_MB", "1")
    synth = kmp.Synth(seed=7, len_mode=1, plants=2, plant_patterns=strings)
    data, offsets = synth.fill_host(0, 12000)  # ~20 MB of mixed sizes: ~20 chunks, every slot reused
    matcher.set_patterns(strings)
    want = finder.find_csr(data, offsets, strings)
    assert np.array_equal(matcher.find_host(data, offsets), want)
    path = os.path.join(DATA, "very_big_udp.pcap")
    pdata, poffsets, _ = oracle.load_pcap_csr(path, "udp")
    pwant = finder.find_csr(pdata, poffsets, strings)
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
        with open(path, "wb") as f:  # UDP frames; a payload is its frame's captured length less the headers
            f.write(struct.pack("<IHHiIII", 0xA1B2C3D4, 2, 4, 0, 0, 262144, 1))
            for p in case:
                frame = bytes(12) + b"\x08\x00" + bytes([0x45, 0, 0, 0, 0, 0, 0, 0, 64, 17]) + bytes(18) + p
                f.write(struct.pack("<IIII", 0, 0, len(frame), len(frame)) + frame)
        counts = oracle.count_csr(data, offsets, strings)
        want = finder.find_csr(data, offsets, strings)
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
    import torch

    synth = kmp.Synth(seed=0xB200, payload_len=1400, plants=2, plant_patterns=strings)
    data, offsets = synth.fill_host(0, 3000)
    matcher.set_patterns(strings)
    d_bytes = torch.zeros(len(data) + 64, dtype=torch.uint8, device="cuda:0")
    d_bytes[: len(data)] = torch.from_numpy(np.array(data))
    d_off = torch.from_numpy(offsets.astype(np.int64)).to("cuda:0")

    def counts():  # (the device form's counts are read once it has finished; tests/test_call_order.py overlaps calls)
        d_counts = torch.zeros(len(strings), dtype=torch.int64, device="cuda:0")
        matcher.count_device(d_bytes.data_ptr(), d_off.data_ptr(), len(offsets) - 1, d_counts.data_ptr(), span=(0, len(data)))
        torch.cuda.synchronize()
        on_device = d_counts.cpu().tolist()
        return matcher.count_host(data, offsets), on_device

    before = counts()
    rec = matcher.find_host(data, offsets)
    device_find(matcher, data, offsets, 10, True)
    assert counts() == before
    assert before[0] == before[1] == oracle.count_csr(data, offsets, strings)
    assert_invariant(before[0], rec, strings)
    matcher.set_engine("perpat")  # finding runs the union engine whatever the engine setting
    try:
        assert np.array_equal(matcher.find_host(data, offsets), rec)
    finally:
        matcher.set_engine("auto")
