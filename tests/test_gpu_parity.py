"""Parity of the CUDA path (through the C ABI of libkmpb200.so) against the oracle and the golden
vectors of the unmodified reference.  Bit-exact: these are integer counts.  Needs a B200."""
import json
import os
import random
import subprocess

import numpy as np
import pytest

from conftest import DATA, GOLDEN, ROOT, golden_runs

import multithreading_string_matching_b200 as kmp

pytestmark = pytest.mark.gpu
ENGINES = ["union", "perpat"]


@pytest.fixture(scope="module")
def matchers():
    ms = {e: kmp.Matcher(0, engine=e) for e in ENGINES}
    yield ms
    for m in ms.values():
        m.close()


@pytest.fixture(scope="module")
def strings(strings_txt):
    return kmp.load_patterns(strings_txt)


def csr(packets):
    offsets = np.zeros(len(packets) + 1, dtype=np.uint64)
    if packets:
        np.cumsum([len(p) for p in packets], out=offsets[1:])
    return np.frombuffer(b"".join(packets) + b"\0" * 16, dtype=np.uint8)[: int(offsets[-1])], offsets


def check_all(matchers, oracle, patterns, packets, engines=ENGINES, label=""):
    data, offsets = csr(packets)
    want = oracle.count_csr(data, offsets, patterns)
    for e in engines:
        m = matchers[e]
        m.set_patterns(patterns)
        got = m.count_host(data, offsets)
        assert got == want, (label, e, [(p, g, w) for p, g, w in zip(patterns, got, want) if g != w][:8])
    return want


# ---- the reference's own fixtures ---------------------------------------------------------------

@pytest.mark.parametrize("engine", ENGINES)
@pytest.mark.parametrize("pcap,proto,expected", golden_runs(), ids=lambda v: v if isinstance(v, str) else "")
def test_bundled_pcaps_bit_exact_vs_serial_c(matchers, strings, engine, pcap, proto, expected):
    """BASELINE config 2: every bundled pcap, output text identical to serial.c's."""
    m = matchers[engine]
    m.set_patterns(strings)
    counts = m.count_pcap(os.path.join(DATA, pcap + ".pcap"), proto, pinned=True)
    assert kmp.format_report(strings, counts) == expected


@pytest.mark.parametrize("pcap,proto,expected", golden_runs(), ids=lambda v: v if isinstance(v, str) else "")
def test_bundled_pcaps_streamed_path(matchers, strings, pcap, proto, expected):
    """The fused ingest + match path (kmpb_pcap_open / kmpb_count_pcap, what bin/kmp_match runs)."""
    m = matchers["union"]
    m.set_patterns(strings)
    counts = m.count_pcap_streamed(os.path.join(DATA, pcap + ".pcap"), proto)
    assert kmp.format_report(strings, counts) == expected


def test_streamed_path_chunks_and_slices(matchers, oracle, strings, tmp_path):
    """Many small staging chunks (the slot ring wraps many times) and rank slices that add up."""
    import sys
    sys.path.insert(0, ROOT)
    import bench
    from multithreading_string_matching_b200 import distributed as kd

    synth = kmp.Synth(seed=23, len_mode=1, plants=2, plant_patterns=strings)
    data, off = synth.fill_host(0, 12_000)
    path = str(tmp_path / "mixed.pcap")
    bench.write_pcap(path, data, off)
    m = matchers["union"]
    m.set_patterns(strings)
    want = oracle.count_csr(data, off, strings)
    os.environ["KMPB_CHUNK_MB"] = "1"
    try:
        assert m.count_pcap_streamed(path) == want
        for world in (2, 3):
            acc = [0] * len(strings)
            for rank in range(world):
                first, count = kd.rank_slice(12_000, rank, world)
                acc = [a + b for a, b in zip(acc, m.count_pcap_streamed(path, first=first, count=count))]
            assert acc == want, world
    finally:
        del os.environ["KMPB_CHUNK_MB"]
    assert m.count_pcap_streamed(path) == want


def _classic_frames(path):
    import struct
    raw = open(path, "rb").read()
    e = "<" if raw[:4] in (b"\xd4\xc3\xb2\xa1", b"\x4d\x3c\xb2\xa1") else ">"
    at, out = 24, []
    while at + 16 <= len(raw):
        caplen = struct.unpack_from(e + "I", raw, at + 8)[0]
        at += 16
        if at + caplen > len(raw):
            break
        out.append(raw[at:at + caplen])
        at += caplen
    return out


@pytest.mark.parametrize("pcap,proto,expected", golden_runs(), ids=lambda v: v if isinstance(v, str) else "")
def test_frames_pushed_one_at_a_time(matchers, strings, pcap, proto, expected):
    """kmpb_stream_*: the live-capture shape (live_openmp_task.c:160-217) fed with the frames of a savefile;
    64 KB batches so that the staging slots are reused many times, a flush in the middle."""
    m = matchers["union"]
    m.set_patterns(strings)
    frames = _classic_frames(os.path.join(DATA, pcap + ".pcap"))
    with m.stream(proto, batch_bytes=65536) as st:
        for f in frames[: len(frames) // 2]:
            st.push(f)
        st.flush()  # partial result; the stream goes on
        for f in frames[len(frames) // 2:]:
            st.push(f)
        counts = st.flush()
    assert kmp.format_report(strings, counts) == expected


def test_cli_output_is_the_reference_output(strings):
    exe = os.path.join(ROOT, "multithreading_string_matching_b200", "bin", "kmp_match")
    for pcap, proto, expected in golden_runs():
        for argv in [[proto], ["1", proto]] + ([[]] if proto == "udp" else []):
            r = subprocess.run([exe, os.path.join(DATA, pcap + ".pcap"), os.path.join(DATA, "strings.txt"), *argv],
                               capture_output=True)
            assert r.returncode == 0, r.stderr
            lines = r.stdout.splitlines(keepends=True)
            assert lines[-1].startswith(b"Elapsed time = ") and lines[-1].endswith(b" seconds\n")
            assert b"".join(lines[:-1]) == expected, (pcap, argv)


def test_bench_dump_outputs_are_the_stream_counts(oracle, strings, tmp_path):
    """bench.py --dump-outputs: the count vector of the last timed step as float64, equal to the oracle's counts on the
    same seeded stream, which bench.py's numpy generator rebuilds on the host."""
    import sys
    import bench

    n = 20_000
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "0", "--packets", str(n),
                        "--no-e2e", "--no-cpu", "--no-sweep", "--no-parity", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    assert json.loads(r.stdout)["steps"] == 2
    got = np.load(str(tmp_path / "counts.npy"))
    data, off = bench.synth_stream(bench.SEED, 0, n, 1400, 2, strings)
    assert got.dtype == np.float64 and got.tolist() == oracle.count_csr(data, off, strings)


def test_integration_snippet_counts(tmp_path):
    """INTEGRATION.md section 1 as a C program (tests/c/integration_snippet.c): overlapping "aa" in "aaaa" = 3, the
    text of a payload ends at its NUL."""
    from test_host import build_integration_snippet
    r = subprocess.run([build_integration_snippet(tmp_path)], capture_output=True, text=True)
    assert r.returncode == 0 and r.stdout == "aa: 3 times!\nhttp: 3 times!\n", (r.stdout, r.stderr)


def test_device_built_prefix_tables(matchers, oracle, strings):
    """kmpb_get_prefix == kmp_prefix (serial.c:217-238): golden vectors + every strings.txt token."""
    vectors = json.load(open(os.path.join(GOLDEN, "kmp_vectors.json")))["vectors"]
    pats = [bytes.fromhex(v["pattern"]) for v in vectors]
    m = matchers["union"]
    m.set_patterns(pats)
    for i, v in enumerate(vectors):
        assert m.prefix(i) == v["pi"], pats[i]
    m.set_patterns(strings)
    for i, p in enumerate(strings):
        assert m.prefix(i) == oracle.kmp_prefix(p)


def test_reference_kmp_vectors(matchers):
    """kmp_matcher (serial.c:190-215) golden vectors: each (text, pattern) pair as a 1-packet batch,
    grouped by pattern set to keep the number of table builds small."""
    vectors = json.load(open(os.path.join(GOLDEN, "kmp_vectors.json")))["vectors"]
    for e in ENGINES:
        m = matchers[e]
        for lo in range(0, len(vectors), 50):
            group = vectors[lo:lo + 50]
            pats = [bytes.fromhex(v["pattern"]) for v in group]
            m.set_patterns(pats)
            data, offsets = csr([bytes.fromhex(v["text"]) for v in group])
            # pattern i is only expected to match its own text; count it over that single packet
            for i, v in enumerate(group):
                one = m.count_host(data[int(offsets[i]):int(offsets[i + 1])], np.array([0, offsets[i + 1] - offsets[i]], dtype=np.uint64))
                assert one[i] == v["count"], (e, pats[i])


# ---- semantics ---------------------------------------------------------------------------------

def test_semantics_overlap_nul_duplicates(matchers, oracle):
    pats = [b"aa", b"ab", b"aa", b"a", b"aaaa", b"b"]
    pkts = [b"aaaa", b"abab\0abab", b"\0aaaa", b"", b"a", b"aaaaaaaaaaaaaaaaaaaaaaaaaaaaaaaaaaaaaaaa", b"ba" * 300]
    want = check_all(matchers, oracle, pats, pkts)
    assert want[0] == want[2] == 3 + 39 and want[1] == 2 + 299


def test_empty_inputs(matchers, oracle):
    check_all(matchers, oracle, [b"x"], [])
    check_all(matchers, oracle, [b"x"], [b"", b"", b""])
    check_all(matchers, oracle, [], [b"abc"])
    check_all(matchers, oracle, [b"abc"], [b"ab", b"c"])  # no match across packets


def test_nul_at_every_position(matchers, oracle):
    """first-NUL truncation (SURVEY fact 1) for a NUL at every offset of a 3-row packet, followed by a
    packet that must be unaffected."""
    pats = [b"ab", b"b", b"abab", b"zz"]
    base = (b"ab" * 700)[:1100]
    pkts = []
    for z in range(0, 1100, 7):
        pkts.append(base[:z] + b"\0" + base[z + 1:])
        pkts.append(b"abab")
    check_all(matchers, oracle, pats, pkts)
    pkts = [base[:z] + b"\0" + base[z + 1:] for z in list(range(0, 40)) + list(range(500, 530)) + list(range(1080, 1100))]
    check_all(matchers, oracle, pats, pkts)


def test_pattern_straddling_every_edge(matchers, oracle):
    """A long self-overlapping pattern placed at every offset around 16-byte group edges, 512-byte row
    edges and packet edges."""
    pat = b"abcabcabcabcabcab"  # 17 bytes: always spans two groups
    pats = [pat, b"abcab", b"bc", b"c", b"cabca"]
    pkts = []
    for start in list(range(0, 40)) + list(range(490, 530)) + list(range(1000, 1040)):
        body = bytearray(b"." * 1100)
        body[start:start + len(pat)] = pat
        pkts.append(bytes(body[:1100]))
    check_all(matchers, oracle, pats, pkts)
    # shifting packet starts: lead packets of every length 0..40 move every later edge
    for lead in range(0, 41, 3):
        check_all(matchers, oracle, pats, [b"x" * lead] + pkts[:20], label="lead%d" % lead)


def test_self_overlap_runs(matchers, oracle):
    pats = [b"a", b"aa", b"aaa", b"a" * 16, b"a" * 17, b"a" * 99, b"rr", b"ara"]
    pkts = [b"a" * n for n in (1, 2, 15, 16, 17, 98, 99, 100, 511, 512, 513, 2048)] + [b"ar" * 600, b"r" * 77]
    check_all(matchers, oracle, pats, pkts)


def test_pattern_lengths_1_to_99(matchers, oracle):
    rng = random.Random(99)
    alpha = b"abcd"
    text = bytes(rng.choice(alpha) for _ in range(6000))
    pats = [text[i * 50:i * 50 + n] for i, n in enumerate(range(1, 100))]
    pkts = [text[:3000], text[3000:], text[100:160], text]
    check_all(matchers, oracle, pats, pkts)


def test_random_batches(matchers, oracle):
    rng = random.Random(20241018)
    lens = [0, 1, 2, 3, 15, 16, 17, 31, 33, 63, 64, 65, 127, 129, 511, 512, 513, 1400, 3000, 9000]
    for trial in range(40):
        alpha = [b"ab", b"abc\0", bytes(range(0x20, 0x7F)), bytes(range(0x20, 0x7F)) + b"\0\0", bytes(range(256))][trial % 5]
        pat_alpha = bytes(b for b in alpha if b) or b"a"
        n_pat = rng.choice([1, 2, 3, 7, 8, 20, 97, 200])
        pats = [bytes(rng.choice(pat_alpha) for _ in range(rng.choice([1, 2, 2, 3, 3, 4, 5, 6, 8, 12, 20, 64])))
                for _ in range(n_pat)]
        n_pkt = rng.choice([1, 2, 5, 40, 300])
        pkts = []
        for _ in range(n_pkt):
            n = rng.choice(lens)
            body = bytearray(rng.choice(alpha) for _ in range(n))
            for _ in range(rng.randint(0, 3)):
                p = rng.choice(pats)
                if len(p) <= n:
                    at = rng.randrange(0, n - len(p) + 1)
                    body[at:at + len(p)] = p
            pkts.append(bytes(body))
        engines = ENGINES if sum(map(len, pkts)) * n_pat < 3e7 else ["union"]
        check_all(matchers, oracle, pats, pkts, engines=engines, label="trial%d" % trial)


def test_many_small_packets_and_item_edges(matchers, oracle):
    """Work items are ~128 KB runs of whole packets: cross many item edges with tiny and odd packets."""
    rng = random.Random(5)
    pats = [b"id", b"ack", b"http", b"content-list", b"NOTIFY", b"rr"]
    pkts = []
    for i in range(9000):
        n = rng.choice([0, 1, 5, 16, 33, 64, 64, 64, 100, 200])
        body = bytearray(rng.choice(b"idackhtpNOTIFYr-_cnsl \0") for _ in range(n))
        pkts.append(bytes(body))
    check_all(matchers, oracle, pats, pkts)
    big = [bytes(rng.choice(b"idackhtp") for _ in range(300_000)) for _ in range(3)]  # packets larger than an item
    check_all(matchers, oracle, pats, big + pkts[:100], engines=["union"])


def test_nul_dense_payloads(matchers, oracle):
    """Binary-looking payloads: most 32-byte groups hold a NUL, so the union engine's rows report from many groups
    and the NUL-only events a later one supersedes are dropped (union_kernel.cu drop_superseded).  What must
    survive: a candidate is alive iff no NUL lies between its packet's start and itself, whatever was dropped."""
    rng = random.Random(77)
    pats = [b"id", b"ack", b"http", b"xy", b"a", b"NOTIFY", b"content-list"]
    for p_nul, n_pkt, top in [(1.0, 40, 3000), (0.97, 60, 2500), (0.7, 80, 2000), (0.3, 80, 2000), (0.1, 120, 1500)]:
        pkts = []
        for _ in range(n_pkt):
            n = rng.randint(0, top)
            body = bytearray(0 if rng.random() < p_nul else rng.choice(b"idackhtpxyNOTIFY") for _ in range(n))
            for _ in range(rng.randint(0, 6)):  # tokens right after packet starts, after NULs and in NUL-free gaps
                p = rng.choice(pats)
                if len(p) <= n:
                    at = rng.choice([0, rng.randrange(0, n - len(p) + 1)])
                    body[at:at + len(p)] = p
            pkts.append(bytes(body))
        check_all(matchers, oracle, pats, pkts, label="p_nul=%g" % p_nul)
    # a NUL-free packet between all-NUL packets, and packets that start inside a NUL-dense row
    pkts = [b"\0" * 5000, b"http id ack " * 40, b"\0" * 37, b"idid", b"\0" * 2048, b"x" * 31 + b"http", b"\0" * 999, b"ackack\0ack"]
    check_all(matchers, oracle, pats, pkts * 7, label="sandwich")


def test_candidate_ring_dense_sparse_and_long(matchers, oracle):
    """The union engine's candidate ring (union_kernel.cu, phase 2 of the resolve step): candidates wait across resolve
    steps until 32 have come together.  Dense candidates -- every byte starts a pattern, more per step than the ring
    holds, so the step falls back to trips of 32 --, a few candidates that are only flushed at the end of the batch,
    and patterns of more than 8 bytes, whose tail is compared against the text in global memory, at every offset of a
    group, across groups, rows and the end of the batch."""
    rng = random.Random(5)
    dense = [b"a", b"aa", b"aaaa", b"aaaaaaaaa", b"ab", b"ba"]
    pkts = [b"a" * rng.randint(0, 700) for _ in range(60)] + [b"ab" * 300, b"a" * 31 + b"\0" + b"a" * 99, b"a" * 5000]
    check_all(matchers, oracle, dense, pkts, label="dense")
    check_all(matchers, oracle, dense, [b"a" * 100_000] * 3, engines=["union"], label="dense, many rows")
    sparse = [b"needle", b"http_decode"]
    check_all(matchers, oracle, sparse, [b"x" * 3000 + b"needle" + b"y" * 2000, b"z" * 100, b"http_decode"], label="sparse")
    long_pats = [b"content-list", b"ignorehosts12345678901234567890", b"0123456789abcdef0123456789abcdef0123456789abcdef0123456789abcdefXYZ"]
    pkts = []
    for p in long_pats:
        for lead in range(0, 70):
            pkts.append(b"." * lead + p)                      # ends with the packet (and once with the batch)
            pkts.append(b"." * lead + p[:-1])                 # one byte short
            pkts.append(b"." * lead + p + b"." * (lead % 5))
    rng.shuffle(pkts)
    check_all(matchers, oracle, long_pats, pkts + [long_pats[2]], label="long")


# ---- synthetic workloads of BASELINE.json ------------------------------------------------------

def test_synthetic_device_resident_stream(matchers, oracle, strings):
    """Config 3 shape at reduced size: generated on the device, identical bits on the host, union
    engine vs oracle on a prefix, additivity over slices, and both engines agreeing on a sample."""
    import torch

    n = 200_000
    synth = kmp.Synth(seed=0xB200, payload_len=1400, plants=2, plant_patterns=strings)
    m = matchers["union"]
    m.set_patterns(strings)
    d_bytes = torch.zeros(n * 1400 + 64, dtype=torch.uint8, device="cuda:0")
    d_off = torch.zeros(n + 1, dtype=torch.int64, device="cuda:0")
    synth.fill_device(m, 0, n, d_bytes.data_ptr(), d_off.data_ptr())
    torch.cuda.synchronize()
    hdata, hoff = synth.fill_host(0, 3000)
    assert np.array_equal(d_bytes[: 3000 * 1400].cpu().numpy(), hdata)
    assert np.array_equal(d_off[:3001].cpu().numpy().astype(np.uint64), hoff)

    def device_counts(first, count):
        d_counts = torch.zeros(len(strings), dtype=torch.int64, device="cuda:0")
        m.count_device(d_bytes.data_ptr(), d_off.data_ptr() + 8 * first, count, d_counts.data_ptr())
        m.count_device(d_bytes.data_ptr(), d_off.data_ptr() + 8 * first, count, d_counts.data_ptr(),
                       span=(first * 1400, (first + count) * 1400))  # accumulates: x2
        torch.cuda.synchronize()
        c = d_counts.cpu().numpy()
        assert (c % 2 == 0).all()
        return (c // 2).tolist()

    whole = device_counts(0, n)
    assert device_counts(0, 3000) == oracle.count_csr(hdata, hoff, strings)
    parts = [device_counts(a, b) for a, b in ((0, 70_001), (70_001, 59_999), (130_000, 70_000))]
    assert whole == [sum(col) for col in zip(*parts)]
    assert sum(whole) >= 2 * n * 0.9  # the planted tokens are found
    p = matchers["perpat"]
    p.set_patterns(strings)
    sample, soff = synth.fill_host(150_000, 2000)
    assert p.count_host(sample, soff) == m.count_host(sample, soff) == oracle.count_csr(sample, soff, strings)


def test_large_pattern_set_tables_in_global_memory(matchers, oracle):
    """700 patterns of up to 99 bytes: the union engine's verification tables (~100 KB) no longer fit behind the row
    rings in shared memory and are read from global memory; one- and two-byte patterns and shared prefixes included."""
    rng = random.Random(4242)
    alpha = b"abcdefgh01"
    pats = [bytes(rng.choice(alpha) for _ in range(rng.choice([1, 2, 2, 3, 4, 5, 8, 9, 13, 40, 41, 64, 99]))) for _ in range(700)]
    pkts = []
    for _ in range(400):
        n = rng.choice([0, 3, 40, 100, 700, 1400, 3000])
        body = bytearray(rng.choice(alpha + b"\0") if rng.random() < 0.02 else rng.choice(alpha) for _ in range(n))
        for _ in range(rng.randint(0, 4)):
            p = rng.choice(pats)
            if len(p) <= n:
                at = rng.randrange(0, n - len(p) + 1)
                body[at:at + len(p)] = p
        pkts.append(bytes(body))
    check_all(matchers, oracle, pats, pkts, engines=["union"], label="700 patterns")


def test_sparse_events_over_many_work_items(matchers, oracle):
    """A batch large enough that every warp of the union engine takes several work items, with events so sparse that
    a warp's list still holds events of the previous item when the next one starts (and, now and then, of the item
    before that: the forced resolve).  The per-pattern engine, which knows nothing of items or events, must agree;
    a prefix is checked against the oracle."""
    import torch

    n, L = 900_000, 1400  # 1.26 GB: ~19 000 items of 64 KB for 4144 warps
    g = torch.Generator(device="cuda:0")
    g.manual_seed(99)
    d_bytes = torch.randint(1, 256, (n * L + 4096,), dtype=torch.uint8, device="cuda:0", generator=g)
    d_bytes[n * L:].zero_()
    # a NUL now and then (one packet in ~60): everything behind it in its packet is dead
    nul_at = torch.randint(0, n * L, (n // 60,), device="cuda:0", generator=g)
    d_bytes[nul_at] = 0
    d_off = torch.arange(0, (n + 1) * L, L, dtype=torch.int64, device="cuda:0")
    pats = [b"\x01\x02", b"ab", b"xyz", b"\xff\xfe\xfd", b"Q"]
    counts = {}
    for e in ENGINES:
        m = matchers[e]
        m.set_patterns(pats)
        d_counts = torch.zeros(len(pats), dtype=torch.int64, device="cuda:0")
        m.count_device(d_bytes.data_ptr(), d_off.data_ptr(), n, d_counts.data_ptr(), span=(0, n * L))
        torch.cuda.synchronize()
        counts[e] = d_counts.cpu().tolist()
    assert counts["union"] == counts["perpat"], counts
    assert min(counts["union"]) > 0
    k = 20_000
    hdata = d_bytes[: k * L].cpu().numpy()
    hoff = np.arange(0, (k + 1) * L, L, dtype=np.uint64)
    m = matchers["union"]
    m.set_patterns(pats)
    assert m.count_host(hdata, hoff) == oracle.count_csr(hdata, hoff, pats)


def test_more_events_per_warp_than_a_16_bit_counter_holds(matchers):
    """Every 32-byte group of the stream raises an event (payloads of one repeated letter, the pattern is that letter
    twice): ~80 000 events per warp of the union engine in one launch.  The event ring's state register must wrap
    without touching its count of pending events (an earlier encoding carried into it after 65 536 events).  The
    counts are known in closed form: a packet of L bytes holds L - 1 overlapping occurrences (serial.c:219 steps to
    pi[q-1] after a match) and L - 2 of the three-letter pattern."""
    import torch

    n, L = 8_600_000, 1400  # 12 GB
    free, _ = torch.cuda.mem_get_info()
    if free < 16 * 2**30:
        pytest.skip("needs 16 GB of device memory")
    d_bytes = torch.full((n * L + 4096,), ord("a"), dtype=torch.uint8, device="cuda:0")
    d_off = torch.arange(0, (n + 1) * L, L, dtype=torch.int64, device="cuda:0")
    pats = [b"aa", b"aaa", b"ab"]
    m = matchers["union"]
    m.set_patterns(pats)
    d_counts = torch.zeros(len(pats), dtype=torch.int64, device="cuda:0")
    m.count_device(d_bytes.data_ptr(), d_off.data_ptr(), n, d_counts.data_ptr(), span=(0, n * L))
    torch.cuda.synchronize()
    assert d_counts.cpu().tolist() == [n * (L - 1), n * (L - 2), 0]
    del d_bytes, d_off
    torch.cuda.empty_cache()


@pytest.mark.parametrize("engine", ["union", "perpat"])
def test_fused_reduce_into_several_vectors(matchers, oracle, strings, engine):
    """kmpb_count_device_span_peers: the counts are added to every vector it is given -- by the union kernel's last
    block, or (per-pattern engine) by the count expansion behind the match kernel, with system-scope atomics in either
    case (on a multi-GPU box the other vectors are peers' memory; here they are local).  bench.py checks the same
    across real GPUs at N > 1 (strong.counts_match_unsplit_stream)."""
    import torch

    synth = kmp.Synth(seed=5, payload_len=700, plants=2, plant_patterns=strings)
    data, off = synth.fill_host(0, 9000)
    want = oracle.count_csr(data, off, strings)
    m = matchers[engine]
    m.set_patterns(strings)
    d_bytes = torch.zeros(len(data) + 4096, dtype=torch.uint8, device="cuda:0")
    d_bytes[: len(data)] = torch.from_numpy(np.ascontiguousarray(data)).cuda()
    d_off = torch.from_numpy(off.astype(np.int64)).cuda()
    vecs = [torch.zeros(len(strings), dtype=torch.int64, device="cuda:0") for _ in range(3)]
    vecs[2] += 7
    for _ in range(2):
        m.count_device_into(d_bytes.data_ptr(), d_off.data_ptr(), 9000, [v.data_ptr() for v in vecs], span=(0, int(off[-1])))
    torch.cuda.synchronize()
    assert vecs[0].cpu().tolist() == [2 * w for w in want]
    assert vecs[1].cpu().tolist() == [2 * w for w in want]
    assert vecs[2].cpu().tolist() == [2 * w + 7 for w in want]
    kmp._lib.check(kmp._lib.lib().kmpb_check_device_errors(m.handle))  # nothing outside the limits was met


def test_mixed_length_stream_host_path(matchers, oracle, strings):
    """Config 5 shape at reduced size through the host (pinned, chunked H2D) entry point."""
    synth = kmp.Synth(seed=11, len_mode=1, plants=2, plant_patterns=strings)
    data, off = synth.fill_host(0, 30_000)
    m = matchers["union"]
    m.set_patterns(strings)
    want = oracle.count_csr(data, off, strings)
    os.environ["KMPB_CHUNK_MB"] = "4"  # force many chunks through the stream pipeline
    try:
        assert m.count_host(data, off) == want
    finally:
        del os.environ["KMPB_CHUNK_MB"]
    assert m.count_host(data, off) == want


def test_pattern_sweep_shapes(matchers, oracle):
    """Config 4 shape at reduced size: n patterns of one length over random [a-z0-9]-ish text."""
    rng = random.Random(4)
    alpha = b"abcdefghijklmnopqrstuvwxyz0123456789"
    text_pk = [bytes(rng.choice(alpha) for _ in range(1400)) for _ in range(300)]
    for n_pat, length in ((1, 4), (16, 8), (64, 16), (256, 4), (256, 64), (128, 32)):
        pats = []
        for i in range(n_pat):
            src = rng.choice(text_pk)
            at = rng.randrange(0, 1400 - length)
            pats.append(src[at:at + length] if i % 2 else bytes(rng.choice(alpha) for _ in range(length)))
        engines = ENGINES if n_pat * length <= 2048 else ["union"]
        check_all(matchers, oracle, pats, text_pk, engines=engines, label="%dx%d" % (n_pat, length))
    # the per-pattern engine tiles pattern sets whose DFAs exceed shared memory
    pats = [bytes(rng.choice(alpha) for _ in range(64)) for _ in range(40)] + [text_pk[0][5:69]]
    check_all(matchers, oracle, pats, text_pk[:40], engines=["perpat"], label="tiled")


def test_sharded_slices_add_up(matchers, oracle, strings):
    """The mpi_dumping.c split on one GPU: each 'rank' matches its own slice of the stream (generated
    independently from the packet counter), the per-rank vectors sum to the whole-stream counts."""
    from multithreading_string_matching_b200 import distributed as kd

    total = 20_001
    synth = kmp.Synth(seed=0xB200, payload_len=1400, plants=2, plant_patterns=strings)
    m = matchers["union"]
    m.set_patterns(strings)
    data, off = synth.fill_host(0, total)
    want = oracle.count_csr(data, off, strings)
    for world in (1, 2, 3, 8):
        acc = [0] * len(strings)
        covered = 0
        for rank in range(world):
            first, count = kd.rank_slice(total, rank, world)
            sd, so = synth.fill_host(first, count)
            acc = [a + b for a, b in zip(acc, m.count_host(sd, so))]
            covered += count
        assert covered == total and acc == want, world
