"""Case-insensitive patterns (KMPB_PAT_NOCASE, Matcher.set_patterns(nocase=...), `kmp_match -i`, `kmp_find -i`) on the
GPU, on both engines and through every count and find form.

Expected answers come from the reference finder (tests/kmpb_reference.py `expected`, with the oracle's counts of each
flag group alongside): a nocase pattern's matches in a text are exactly the case-sensitive matches of the folded
pattern in the folded text.  tests/test_tables_nocase.py checks that derivation against a naive finder."""
import ctypes
import os
import random
import subprocess

import numpy as np
import pytest

from conftest import DATA, golden_runs
from kmpb_harness import (FIND, FIND_FORMS, FIND_HOST_FORMS, MATCH, STRINGS, DeviceBatch, check_forms, engines,  # noqa: F401
                          pcap_frames)
from kmpb_reference import LETTERS, ORDER, as_tuples, csr, expected, fold, gate_kept, planted_packets

import multithreading_string_matching_b200 as kmp


@pytest.mark.gpu
def test_semantics(engines, oracle):
    got = check_forms(engines, [b"aA"], *csr([b"AaAa"]), True, oracle=oracle, forms=FIND_FORMS)[1]
    assert as_tuples(got) == [(0, 0, 0), (0, 1, 0), (0, 2, 0)]
    # one distinct pattern: every listing gets the full count, the records carry the first index
    got = check_forms(engines, [b"Ack", b"ACK", b"ack"], *csr([b"ack ACK aCk"]), True, oracle=oracle, forms=FIND_FORMS)[1]
    assert as_tuples(got) == [(0, 0, 0), (0, 4, 0), (0, 8, 0)]
    assert engines[0].count_host(*csr([b"ack ACK aCk"])) == [3, 3, 3]
    # case-sensitive "ack" and nocase "ACK" are two: one occurrence of "ack" yields a record for each
    got = check_forms(engines, [b"ack", b"ACK"], *csr([b"ack Ack"]), [False, True], oracle=oracle, forms=FIND_FORMS)[1]
    assert as_tuples(got) == [(0, 0, 0), (0, 0, 1), (0, 4, 1)]
    # a token without letters behaves as case-sensitive; letterless text counts as it does case-sensitively
    check_forms(engines, [b"12", b"-/:", b"@@"], *csr([b"12 -/: @@@ 1@2"]), True, oracle=oracle, forms=FIND_FORMS)
    pats = [b"ab", b"x", b"ab12", b"http://"]
    pkts = [bytes(random.Random(k).choice(b"0123456789-/:@[ ") for _ in range(200)) for k in range(20)]
    data, offsets = csr(pkts)
    engines[0].set_patterns(pats)
    cs = engines[0].count_host(data, offsets)
    check_forms(engines, pats, *csr(pkts), True, oracle=oracle, forms=FIND_FORMS)
    assert engines[0].count_host(data, offsets) == cs
    # the bytes that differ from another in bit 5 only and are not letters never fold
    got = check_forms(engines, [b"@[\\]^_", b"\xc1", b"\xdf", b"@", b"_"],
                      *csr([b"`{|}~\x7f", b"\xe1\xff`\x7f", b"@[\\]^_ \xc1\xdf @ _"]), True, oracle=oracle, forms=FIND_FORMS)[1]
    assert as_tuples(got) == [(2, 0, 0), (2, 0, 3), (2, 5, 4), (2, 7, 1), (2, 8, 2), (2, 10, 3), (2, 12, 4)]
    # the text ends at the first NUL; matches lie inside one packet
    got = check_forms(engines, [b"AB", b"b"], *csr([b"abAB\0ab", b"\0AB", b"xa", b"Bab"]), True, oracle=oracle, forms=FIND_FORMS)[1]
    assert as_tuples(got) == [(0, 0, 0), (0, 1, 1), (0, 2, 0), (0, 3, 1), (3, 0, 1), (3, 1, 0), (3, 2, 1)]


@pytest.mark.gpu
def test_lengths_1_to_99_case_flipped_at_every_position(engines, oracle):
    rng = random.Random(1999)
    pats = [bytes(rng.choice(b"abcxyz") for _ in range(m)) for m in range(1, 100)]
    pkts = []
    for p in pats:
        for j in range(len(p)):  # gate key (0-1), gate bit (2), record bytes 3-7, tail (8+), last byte
            q = bytearray(p)
            q[j] ^= 0x20
            pkts.append(b"-" * (j % 5) + bytes(q) + b"-" * (j % 3))
        pkts.append(p.upper())
    check_forms(engines, pats, *csr(pkts), True, label="flipped", oracle=oracle, forms=FIND_FORMS)
    alphabet = b"abcxyzABCXYZ-"
    mixed = [bytes(rng.choice(b"abcxyzABCXYZ") for _ in range(rng.randint(1, 40))) for _ in range(60)]
    planted = planted_packets(rng, mixed, alphabet, 400, 160)
    planted = [bytes(c ^ 0x20 if c in LETTERS and rng.random() < 0.5 else c for c in p) for p in planted]
    check_forms(engines, mixed, *csr(planted), [rng.random() < 0.7 for _ in mixed], label="planted", oracle=oracle,
                forms=FIND_FORMS)


@pytest.mark.gpu
def test_case_sensitive_and_nocase_claim_the_same_bytes(engines, oracle):
    pats = [b"A", b"a", b"b", b"B", b"Ab", b"aB", b"xYz", b"XYZ", b"ack", b"ACK", b"ackACKack", b"ACKackACK"]
    nocase = [False, True, False, True, False, True, False, True, False, True, False, True]
    pkts = [b"aAbB", b"AbaBABab", b"xyzXYZxYz", b"ack ACK Ack", b"ackackackACKACKACKackACKack", b"A", b"b"]
    got = check_forms(engines, pats, *csr(pkts), nocase, oracle=oracle, forms=FIND_FORMS)[1]
    assert (0, 0, 0) not in as_tuples(got) and (5, 0, 0) in as_tuples(got) and (5, 0, 1) in as_tuples(got)


@pytest.mark.gpu
def test_table_placement(engines, oracle):
    rng = random.Random(31)
    # gate kept, probe tables in shared memory
    small = [b"host", b"Accept", b"xy"]
    assert gate_kept(small, [True] * 3)
    check_forms(engines, small, *csr(planted_packets(rng, small, b"hostacepxyHOSTACEPXY ", 300, 200)), True, oracle=oracle,
                forms=FIND_FORMS)
    # the gate lost to the case variants (the same set case-sensitive keeps it)
    two = sorted({bytes(rng.choice(b"abcdefghijklmnopqrstuvwxyz") for _ in range(2)) for _ in range(150)})[:120]
    assert gate_kept(two, [False] * len(two)) and not gate_kept(two, [True] * len(two))
    alpha = b"abcdefghijklmnopqrstuvwxyzABCDEFGHIJKLMNOPQRSTUVWXYZ "
    check_forms(engines, two, *csr(planted_packets(rng, two, alpha, 300, 200)), True, label="no gate", oracle=oracle,
                forms=FIND_FORMS)
    # probe tables in global memory (about 700 nocase patterns: several records each)
    many = [bytes(rng.choice(alpha[:-1]) for _ in range(rng.randint(3, 30))) for _ in range(700)]
    check_forms(engines, many, *csr(planted_packets(rng, many, alpha, 400, 300)), True, label="global vtab", oracle=oracle,
                forms=FIND_FORMS)
    # counters in global memory (more than 4096 distinct patterns)
    lots = sorted({bytes(rng.choice(b"abcdefgh") for _ in range(rng.randint(4, 9))) for _ in range(6000)})
    assert len(lots) > 4096
    check_forms(engines, lots, *csr(planted_packets(rng, lots, b"abcdefghABCDEFGH", 400, 300)),
                [i % 3 != 0 for i in range(len(lots))], label="global counts", oracle=oracle, forms=FIND_FORMS)


@pytest.mark.gpu
def test_device_count_forms_and_prefix(engines, oracle):
    import torch

    union, perpat = engines
    rng = random.Random(5)
    pats = [b"Host", b"http", b"HTTP", b"a", b"Content-Type", b"ab", b"xyzzy-plugh-forty-two"]
    nocase = [True, False, True, True, True, False, True]
    pkts = planted_packets(rng, pats, b"hostpcnteaybzxHOSTPCNTEAYBZX-: ", 2000, 400)
    pkts = [bytes(c ^ 0x20 if c in LETTERS and rng.random() < 0.3 else c for c in p) for p in pkts]
    data, offsets = csr(pkts)
    want, want_rec, _ = expected(pats, data, offsets, nocase, oracle=oracle)
    batch = DeviceBatch(data, offsets)
    for m in (union, perpat):
        m.set_patterns(pats, nocase)
        d_counts = torch.zeros(len(pats), dtype=torch.int64, device="cuda:0")
        m.count_device(batch.d_bytes.data_ptr(), batch.d_off.data_ptr(), len(pkts), d_counts.data_ptr(), span=(0, len(data)))
        m.count_device_into(batch.d_bytes.data_ptr(), batch.d_off.data_ptr(), len(pkts), [d_counts.data_ptr()], (0, len(data)))
        torch.cuda.synchronize()
        assert d_counts.cpu().tolist() == [2 * c for c in want]
        for i, p in enumerate(pats):
            assert m.prefix(i) == oracle.kmp_prefix(fold(p) if nocase[i] else p)
    # one record short: the total is exact, what is written is a subset, the canary stays
    union.set_patterns(pats, nocase)
    rec, total, ok = batch.find(union, len(want_rec) - 1, True)
    assert total == len(want_rec) and ok and len(rec) == len(want_rec) - 1
    assert set(as_tuples(rec)) <= set(as_tuples(want_rec))


@pytest.mark.gpu
@pytest.mark.parametrize("pcap,proto", [(p, q) for p, q, _ in golden_runs()])
def test_bundled_pcaps_every_form_and_the_command_lines(engines, oracle, pcap, proto):
    union, perpat = engines
    path = os.path.join(DATA, pcap + ".pcap")
    tokens = oracle.load_patterns(STRINGS)
    data, offsets, _ = oracle.load_pcap_csr(path, proto)
    want_counts, want, _ = expected(tokens, data, offsets, nocase=True, oracle=oracle)
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
    assert np.array_equal(got[ORDER].astype(kmp.MATCH_DTYPE), want)
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
def test_switching_sets_and_flags(engines, oracle):
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
def test_randomised_mixed_sets(engines, oracle):
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
        check_forms(engines, pats, *csr(pkts), nocase, label=trial, oracle=oracle,
                    forms=FIND_FORMS if trial % 10 == 0 else FIND_HOST_FORMS)
