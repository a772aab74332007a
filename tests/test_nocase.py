"""Case-insensitive patterns (KMPB_PAT_NOCASE, Matcher.set_patterns(nocase=...), `kmp_match -i`, `kmp_find -i`) on the
GPU, on both engines and through every count and find form.

Expected answers come from the unchanged oracle and reference finder: a nocase pattern's matches in a text are exactly
the case-sensitive matches of the folded pattern in the folded text (folding never creates or moves a NUL).  So the
case-sensitive patterns are run on the original payloads, the nocase ones, folded, on folded copies, and the records
are renumbered to the first index of each distinct (folded bytes, flag) pattern.  tests/test_tables_nocase.py checks
that derivation against a naive case-insensitive finder."""
import ctypes
import os
import random
import subprocess

import numpy as np
import pytest

from conftest import DATA, ROOT, golden_runs
from test_find import FIND, RefFinder, as_tuples, csr, device_find, pcap_frames
from test_prefix_gate import GATE_MUL, planted_packets

import multithreading_string_matching_b200 as kmp

MATCH = os.path.join(ROOT, "multithreading_string_matching_b200", "bin", "kmp_match")
STRINGS = os.path.join(DATA, "strings.txt")
_FOLD = bytes(c + 32 if 0x41 <= c <= 0x5A else c for c in range(256))
LETTERS = set(range(0x41, 0x5B)) | set(range(0x61, 0x7B))


def fold(b):
    return bytes(b).translate(_FOLD)


def first_index_nc(patterns, nocase):
    """file-order index -> lowest index of the same distinct pattern: equal flag, equal bytes (after folding when nocase)"""
    seen = {}
    return [seen.setdefault((fold(p) if n else bytes(p), bool(n)), i) for i, (p, n) in enumerate(zip(patterns, nocase))]


def expected(oracle, finder, patterns, nocase, data, offsets):
    """(counts, sorted records) of a mixed set from the oracle and the reference finder"""
    patterns = [bytes(p) for p in patterns]
    firsts = first_index_nc(patterns, nocase)
    data = np.ascontiguousarray(data, dtype=np.uint8)
    folded = np.frombuffer(fold(data.tobytes()), dtype=np.uint8)
    counts, parts = [0] * len(patterns), []
    for want_nc, text in ((False, data), (True, folded)):
        idx = [i for i in range(len(patterns)) if bool(nocase[i]) == want_nc]
        if not idx:
            continue
        sub = [fold(patterns[i]) if want_nc else patterns[i] for i in idx]
        for i, c in zip(idx, oracle.count_csr(text, offsets, sub)):
            counts[i] = c
        r = finder.find_csr(text, offsets, sub)
        r["pattern"] = np.array([firsts[i] for i in idx], dtype=np.uint32)[r["pattern"].astype(np.int64)]
        parts.append(r)
    rec = np.concatenate(parts) if parts else np.zeros(0, dtype=kmp.MATCH_DTYPE)
    return counts, np.sort(rec, order=["packet", "offset", "pattern"])


def naive_nocase_find(packets, patterns, nocase):
    """sorted (packet, offset, pattern) straight from the definition"""
    firsts = first_index_nc(patterns, nocase)
    out = []
    for k, payload in enumerate(packets):
        text = payload.split(b"\0", 1)[0]
        for i, (p, n) in enumerate(zip(patterns, nocase)):
            if firsts[i] != i:
                continue
            t, q = (fold(text), fold(p)) if n else (text, p)
            out += [(k, s, i) for s in range(len(t) - len(q) + 1) if t[s:s + len(q)] == q]
    return sorted(out)


def gate_kept(patterns, nocase):
    """whether automaton.c build_gate builds a gate for this set (the variants of a nocase key count as keys)"""
    u = sorted({(fold(p) if n else bytes(p), bool(n)) for p, n in zip(patterns, nocase)})
    keys, last = 0, None
    for p, n in u:
        vs = [i for i in range(min(len(p), 2)) if n and p[i] in LETTERS]
        if len(p) == 1:
            keys += 256 << len(vs)
        elif n:
            keys += 1 << len(vs)
        else:
            keys += p[:2] != last
            last = p[:2]
    log_w = 5
    while (1 << log_w) < 1024 and (1 << log_w) < 16 * keys:
        log_w += 1
    shift = 32 - log_w
    g = [0] * (1 << log_w)
    for p, n in u:
        for v0 in ([p[0], p[0] ^ 0x20] if n and p[0] in LETTERS else [p[0]]):
            if len(p) == 1:
                for c in range(256):
                    g[(((v0 | c << 8) * GATE_MUL) & 0xFFFFFFFF) >> shift] = 0xFFFFFFFF
                continue
            for v1 in ([p[1], p[1] ^ 0x20] if n and p[1] in LETTERS else [p[1]]):
                w = (((v0 | v1 << 8) * GATE_MUL) & 0xFFFFFFFF) >> shift
                g[w] |= 0xFFFFFFFF if len(p) == 2 else 0x80000000 >> (p[2] & 31)
    return bool(u) and 8 * sum(bin(w).count("1") for w in g) <= 32 * len(g)


@pytest.fixture(scope="module")
def finder(tmp_path_factory):
    return RefFinder(str(tmp_path_factory.mktemp("kmp_find_ref_nc")))


@pytest.fixture(scope="module")
def engines():
    u, p = kmp.Matcher(0, engine="union"), kmp.Matcher(0, engine="perpat")
    yield u, p
    u.close()
    p.close()


def check(engines, oracle, finder, patterns, nocase, packets, label="", device=True):
    """both engines' counts and every in-memory find form against the expected answers; returns the records"""
    union, perpat = engines
    if isinstance(nocase, bool):
        nocase = [nocase] * len(patterns)
    data, offsets = csr(packets)
    want_counts, want = expected(oracle, finder, patterns, nocase, data, offsets)
    union.set_patterns(patterns, nocase)
    perpat.set_patterns(patterns, nocase)
    assert union.nocase == list(nocase)
    assert union.count_host(data, offsets) == want_counts, label
    assert perpat.count_host(data, offsets) == want_counts, label
    got = union.find_host(data, offsets)
    if not np.array_equal(got, want):
        w, g = set(as_tuples(want)), set(as_tuples(got))
        raise AssertionError((label, len(want), len(got), sorted(w - g)[:5], sorted(g - w)[:5]))
    if device and len(packets) and len(want):
        rec, total, ok = device_find(union, data, offsets, len(want), True)
        assert total == len(want) and ok and np.array_equal(rec, want), label
        rec, total, ok = device_find(union, data, offsets, len(want), False)
        assert total == len(want) and ok and np.array_equal(np.sort(rec, order=["packet", "offset", "pattern"]), want), label
    return want


@pytest.mark.gpu
def test_semantics(engines, oracle, finder):
    got = check(engines, oracle, finder, [b"aA"], True, [b"AaAa"])
    assert as_tuples(got) == [(0, 0, 0), (0, 1, 0), (0, 2, 0)]
    # one distinct pattern: every listing gets the full count, the records carry the first index
    got = check(engines, oracle, finder, [b"Ack", b"ACK", b"ack"], True, [b"ack ACK aCk"])
    assert as_tuples(got) == [(0, 0, 0), (0, 4, 0), (0, 8, 0)]
    assert engines[0].count_host(*csr([b"ack ACK aCk"])) == [3, 3, 3]
    # case-sensitive "ack" and nocase "ACK" are two: one occurrence of "ack" yields a record for each
    got = check(engines, oracle, finder, [b"ack", b"ACK"], [False, True], [b"ack Ack"])
    assert as_tuples(got) == [(0, 0, 0), (0, 0, 1), (0, 4, 1)]
    # a token without letters behaves as case-sensitive; letterless text counts as it does case-sensitively
    check(engines, oracle, finder, [b"12", b"-/:", b"@@"], True, [b"12 -/: @@@ 1@2"])
    pats = [b"ab", b"x", b"ab12", b"http://"]
    pkts = [bytes(random.Random(k).choice(b"0123456789-/:@[ ") for _ in range(200)) for k in range(20)]
    data, offsets = csr(pkts)
    engines[0].set_patterns(pats)
    cs = engines[0].count_host(data, offsets)
    assert check(engines, oracle, finder, pats, True, pkts) is not None and engines[0].count_host(data, offsets) == cs
    # the bytes that differ from another in bit 5 only and are not letters never fold
    got = check(engines, oracle, finder, [b"@[\\]^_", b"\xc1", b"\xdf", b"@", b"_"], True,
                [b"`{|}~\x7f", b"\xe1\xff`\x7f", b"@[\\]^_ \xc1\xdf @ _"])
    assert as_tuples(got) == [(2, 0, 0), (2, 0, 3), (2, 5, 4), (2, 7, 1), (2, 8, 2), (2, 10, 3), (2, 12, 4)]
    # the text ends at the first NUL; matches lie inside one packet
    got = check(engines, oracle, finder, [b"AB", b"b"], True, [b"abAB\0ab", b"\0AB", b"xa", b"Bab"])
    assert as_tuples(got) == [(0, 0, 0), (0, 1, 1), (0, 2, 0), (0, 3, 1), (3, 0, 1), (3, 1, 0), (3, 2, 1)]


@pytest.mark.gpu
def test_lengths_1_to_99_case_flipped_at_every_position(engines, oracle, finder):
    rng = random.Random(1999)
    pats = [bytes(rng.choice(b"abcxyz") for _ in range(m)) for m in range(1, 100)]
    pkts = []
    for p in pats:
        for j in range(len(p)):  # gate key (0-1), gate bit (2), record bytes 3-7, tail (8+), last byte
            q = bytearray(p)
            q[j] ^= 0x20
            pkts.append(b"-" * (j % 5) + bytes(q) + b"-" * (j % 3))
        pkts.append(p.upper())
    check(engines, oracle, finder, pats, True, pkts, label="flipped")
    alphabet = b"abcxyzABCXYZ-"
    mixed = [bytes(rng.choice(b"abcxyzABCXYZ") for _ in range(rng.randint(1, 40))) for _ in range(60)]
    planted = planted_packets(rng, mixed, alphabet, 400, 160)
    planted = [bytes(c ^ 0x20 if c in LETTERS and rng.random() < 0.5 else c for c in p) for p in planted]
    check(engines, oracle, finder, mixed, [rng.random() < 0.7 for _ in mixed], planted, label="planted")


@pytest.mark.gpu
def test_case_sensitive_and_nocase_claim_the_same_bytes(engines, oracle, finder):
    pats = [b"A", b"a", b"b", b"B", b"Ab", b"aB", b"xYz", b"XYZ", b"ack", b"ACK", b"ackACKack", b"ACKackACK"]
    nocase = [False, True, False, True, False, True, False, True, False, True, False, True]
    pkts = [b"aAbB", b"AbaBABab", b"xyzXYZxYz", b"ack ACK Ack", b"ackackackACKACKACKackACKack", b"A", b"b"]
    got = check(engines, oracle, finder, pats, nocase, pkts)
    assert (0, 0, 0) not in as_tuples(got) and (5, 0, 0) in as_tuples(got) and (5, 0, 1) in as_tuples(got)


@pytest.mark.gpu
def test_table_placement(engines, oracle, finder):
    rng = random.Random(31)
    # gate kept, probe tables in shared memory
    small = [b"host", b"Accept", b"xy"]
    assert gate_kept(small, [True] * 3)
    check(engines, oracle, finder, small, True, planted_packets(rng, small, b"hostacepxyHOSTACEPXY ", 300, 200))
    # the gate lost to the case variants (the same set case-sensitive keeps it)
    two = sorted({bytes(rng.choice(b"abcdefghijklmnopqrstuvwxyz") for _ in range(2)) for _ in range(150)})[:120]
    assert gate_kept(two, [False] * len(two)) and not gate_kept(two, [True] * len(two))
    alpha = b"abcdefghijklmnopqrstuvwxyzABCDEFGHIJKLMNOPQRSTUVWXYZ "
    check(engines, oracle, finder, two, True, planted_packets(rng, two, alpha, 300, 200), label="no gate")
    # probe tables in global memory (about 700 nocase patterns: several records each)
    many = [bytes(rng.choice(alpha[:-1]) for _ in range(rng.randint(3, 30))) for _ in range(700)]
    check(engines, oracle, finder, many, True, planted_packets(rng, many, alpha, 400, 300), label="global vtab")
    # counters in global memory (more than 4096 distinct patterns)
    lots = sorted({bytes(rng.choice(b"abcdefgh") for _ in range(rng.randint(4, 9))) for _ in range(6000)})
    assert len(lots) > 4096
    check(engines, oracle, finder, lots, [i % 3 != 0 for i in range(len(lots))],
          planted_packets(rng, lots, b"abcdefghABCDEFGH", 400, 300), label="global counts")


@pytest.mark.gpu
def test_device_count_forms_and_prefix(engines, oracle, finder):
    import torch

    union, perpat = engines
    rng = random.Random(5)
    pats = [b"Host", b"http", b"HTTP", b"a", b"Content-Type", b"ab", b"xyzzy-plugh-forty-two"]
    nocase = [True, False, True, True, True, False, True]
    pkts = planted_packets(rng, pats, b"hostpcnteaybzxHOSTPCNTEAYBZX-: ", 2000, 400)
    pkts = [bytes(c ^ 0x20 if c in LETTERS and rng.random() < 0.3 else c for c in p) for p in pkts]
    data, offsets = csr(pkts)
    want, _ = expected(oracle, finder, pats, nocase, data, offsets)
    d_bytes = torch.zeros(len(data) + 64, dtype=torch.uint8, device="cuda:0")
    d_bytes[: len(data)] = torch.from_numpy(np.array(data))
    d_off = torch.from_numpy(offsets.astype(np.int64)).to("cuda:0")
    for m in (union, perpat):
        m.set_patterns(pats, nocase)
        d_counts = torch.zeros(len(pats), dtype=torch.int64, device="cuda:0")
        m.count_device(d_bytes.data_ptr(), d_off.data_ptr(), len(pkts), d_counts.data_ptr(), span=(0, len(data)))
        m.count_device_into(d_bytes.data_ptr(), d_off.data_ptr(), len(pkts), [d_counts.data_ptr()], (0, len(data)))
        torch.cuda.synchronize()
        assert d_counts.cpu().tolist() == [2 * c for c in want]
        for i, p in enumerate(pats):
            assert m.prefix(i) == oracle.kmp_prefix(fold(p) if nocase[i] else p)
    # one record short: the total is exact, what is written is a subset, the canary stays
    union.set_patterns(pats, nocase)
    _, want_rec = expected(oracle, finder, pats, nocase, data, offsets)
    rec, total, ok = device_find(union, data, offsets, len(want_rec) - 1, True)
    assert total == len(want_rec) and ok and len(rec) == len(want_rec) - 1
    assert set(as_tuples(rec)) <= set(as_tuples(want_rec))


@pytest.mark.gpu
@pytest.mark.parametrize("pcap,proto", [(p, q) for p, q, _ in golden_runs()])
def test_bundled_pcaps_every_form_and_the_command_lines(engines, oracle, finder, pcap, proto):
    union, perpat = engines
    path = os.path.join(DATA, pcap + ".pcap")
    tokens = oracle.load_patterns(STRINGS)
    data, offsets, _ = oracle.load_pcap_csr(path, proto)
    want_counts, want = expected(oracle, finder, tokens, [True] * len(tokens), data, offsets)
    union.set_patterns(tokens, nocase=True)
    perpat.set_patterns(tokens, nocase=True)
    for m in (union, perpat):
        assert m.count_pcap(path, proto) == want_counts
        assert m.count_pcap_streamed(path, proto) == want_counts
    frames = pcap_frames(path)
    with union.stream(proto, batch_bytes=1 << 16) as st:
        for f in frames:
            st.push(f)
        assert st.flush() == want_counts
    got = union.find_pcap(path, proto)
    assert np.array_equal(got[["packet", "offset", "pattern"]].astype(kmp.MATCH_DTYPE), want)
    accepted = [i for i, f in enumerate(frames) if oracle.extract(f, proto) is not None]
    assert got["frame"].tolist() == [accepted[k] for k in want["packet"].tolist()]
    # the command lines: the report lists each token as spelled, with its case-insensitive count
    report = oracle.format_report(tokens, want_counts)
    for argv in ([proto], ["1", proto]):
        r = subprocess.run([MATCH, "-i", path, STRINGS, *argv], capture_output=True)
        assert r.returncode == 0, r.stderr
        lines = r.stdout.splitlines(keepends=True)
        assert lines[-1].startswith(b"Elapsed time = ") and b"".join(lines[:-1]) == report, argv
    r = subprocess.run([FIND, "-i", path, STRINGS, proto], capture_output=True)
    assert r.returncode == 0, r.stderr
    lines = ["%d %d %s" % (accepted[k] + 1, o, tokens[p].decode("latin-1")) for k, o, p in as_tuples(want)]
    assert r.stdout.decode("latin-1").splitlines() == lines


@pytest.mark.gpu
def test_switching_sets_and_flags(engines, oracle, finder):
    union, _ = engines
    tokens = oracle.load_patterns(STRINGS)
    path = os.path.join(DATA, "big_udp.pcap")
    data, offsets, _ = oracle.load_pcap_csr(path, "udp")
    cs = oracle.count_csr(data, offsets, tokens)
    union.set_patterns(tokens, nocase=True)
    nc = union.count_host(data, offsets)
    assert all(n >= c for n, c in zip(nc, cs)) and nc != cs
    union.set_patterns(tokens)
    assert union.count_host(data, offsets) == cs and union.nocase == [False] * len(tokens)
    # flags == NULL is the plain call; an unknown bit is refused, naming the pattern
    blob, off = kmp.pack_patterns(tokens)
    lib = kmp.lib()
    u8p, u32p = ctypes.POINTER(ctypes.c_uint8), ctypes.POINTER(ctypes.c_uint32)
    assert lib.kmpb_set_patterns_ex(union.handle, blob.ctypes.data_as(u8p), off.ctypes.data_as(u32p), len(tokens), None) == 0
    assert union.count_host(data, offsets) == cs
    flags = np.zeros(len(tokens), dtype=np.uint8)
    flags[3] = 4
    rc = lib.kmpb_set_patterns_ex(union.handle, blob.ctypes.data_as(u8p), off.ctypes.data_as(u32p), len(tokens),
                                  flags.ctypes.data_as(u8p))
    assert rc == -1 and b"pattern 3" in lib.kmpb_last_error()
    with pytest.raises(ValueError):
        union.set_patterns(tokens, nocase=[True])


@pytest.mark.gpu
def test_randomised_mixed_sets(engines, oracle, finder):
    rng = random.Random(0xCA5E)
    alphas = [b"aAbB", b"abcABC@`[{", b"aAzZ@`[{\\|]}^~_\x7f\xc1\xe1\xdf\xff", bytes(range(0x20, 0x7F)), bytes(range(1, 256))]
    for trial in range(300):
        alpha = alphas[trial % len(alphas)]
        pats = [bytes(rng.choice(alpha) for _ in range(rng.choice([1, 2, 3, 4, 5, 8, 9, 12, 20, 40])))
                for _ in range(rng.choice([1, 2, 5, 12, 40]))]
        if len(pats) > 1 and trial % 4 == 0:
            pats.append(pats[0].swapcase())
        nocase = [rng.random() < 0.6 for _ in pats]
        size = rng.choice([3, 30, 200, 1500])
        text = alpha + b"\0" * (trial % 3 == 0)
        pkts = [bytes(rng.choice(text) for _ in range(rng.randint(0, size))) for _ in range(rng.randint(1, 30))]
        pkts = [bytes(c ^ 0x20 if c in LETTERS and rng.random() < 0.5 else c for c in p) for p in pkts]
        check(engines, oracle, finder, pats, nocase, pkts, label=trial, device=trial % 10 == 0)
