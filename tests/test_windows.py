"""Position windows (kmpb_set_patterns_win, Matcher.set_patterns(window=...), `-w LO:HI` of the command lines) on the
GPU: both engines, every count, find and select form.

Expected answers come from the reference finder (tests/kmpb_reference.py `expected`): the records of each pattern
without its window, those whose offset lies in the pattern's window, re-keyed to the lowest index of equal (bytes,
flag, window).  tests/test_tables_windows.py checks that derivation against a naive finder."""
import os
import random
import subprocess

import numpy as np
import pytest

from conftest import DATA
from kmpb_harness import (DEVICE_FORMS, FIND, HOST_FORMS, MATCH, PCAPS, SELECT, STRINGS, DeviceBatch, check_forms, engines,  # noqa: F401
                          pcap_frames, udp_frame, write_pcap)
from kmpb_reference import ORDER, as_tuples, csr, expected

import multithreading_string_matching_b200 as kmp


@pytest.mark.gpu
def test_window_edges_and_semantics(engines):
    A = ord("a")
    cases = [
        # hits at lo - 1, lo, hi, hi + 1; lo = hi
        ([b"xab" + b"ab" * 6], [b"ab"], [(3, 9)]),
        ([b"xxxxab", b"xxxab", b"xxxxxab"], [b"ab"], [(4, 4)]),
        # a match that ends exactly at the packet's end, one that would run past it
        ([b"xxGET", b"xxxGE", b"xxxxGET"], [b"GET"], [(0, 3)]),
        # a NUL inside, before and after the match
        ([b"xxab", b"x\0ab", b"xxa\0b", b"xxab\0"], [b"ab"], [(2, 2)]),
        # overlaps inside a window
        ([b"aaaa"], [b"aa"], [(1, 2)]),
        # the same bytes under different windows, and alongside an unwindowed copy (duplicates keep the first index)
        ([b"ab" * 10, b"xab"], [b"ab", b"ab", b"ab", b"ab", b"ab"], [(0, 0), None, (0, 5), (0, 0), (2, 2)]),
        # empty packets, packets shorter than lo
        ([b"", b"ab", b"", b"xxab", b"xxxxxxxxab"], [b"ab", b"b"], [(8, 20), (9, 9)]),
        # every pattern windowed, one-byte patterns
        ([bytes([A]) * 50, b"b" * 3], [b"a", b"b"], [(10, 19), (0, 0)]),
    ]
    for pkts, pats, win in cases:
        check_forms(engines, pats, *csr(pkts), False, win, label=(pats, win))
    # nocase together with a window, and a case-sensitive copy under another window
    pkts = [b"xGeT gEt GET get", b"GETget", b"\0GET"]
    check_forms(engines, [b"get", b"GET", b"get"], *csr(pkts), [True, False, False], [(0, 5), (0, 20), None],
                label="nocase")
    check_forms(engines, [b"get", b"Get"], *csr(pkts), True, (4, 8), label="nocase all windowed")


@pytest.mark.gpu
def test_pattern_lengths_and_long_windows(engines):
    rng = random.Random(5)
    for m in (1, 2, 3, 8, 9, 99):
        p = bytes(rng.choice(b"abc") for _ in range(m))
        pkts = [bytes(rng.choice(b"abc") for _ in range(rng.randint(0, 400))) for _ in range(30)]
        pkts += [p * 5, b"x" * 7 + p, b"x" * 300 + p + p]
        check_forms(engines, [p, b"ab", p], *csr(pkts), [False, False, True], [(0, 7), None, (5, 320)], label=m)
    # hi = 65535 in a 70 KB packet, starts on both sides of it and at tile edges
    big = bytearray(b"y" * 70000)
    for o in (100, 1023, 1024, 2047, 65535, 65536, 69998):
        big[o:o + 2] = b"ab"
    check_forms(engines, [b"ab", b"yyab"], *csr([bytes(big), b"ab"]), False, (100, 65535), label="65535")
    check_forms(engines, [b"ab", b"y"], *csr([bytes(big)]), False, [(0, 65535), None], label="65535 mixed")
    # a NUL in a tile's lookahead: the next tile still tests the starts before it
    edge = bytearray(b"y" * 3000)
    edge[1025:1027] = b"ab"
    edge[1040] = 0
    check_forms(engines, [b"ab", b"yyab"], *csr([bytes(edge)]), False, (0, 2000), label="nul in the lookahead")
    # a NUL far into the head ends the text for every later tile
    big[40000] = 0
    check_forms(engines, [b"ab"], *csr([bytes(big)]), False, (0, 65535), label="nul at 40000")


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["mixed", "all_windowed"])
def test_every_form(engines, kind, tmp_path):
    tokens = kmp.load_patterns(STRINGS)
    rng = random.Random(11)
    pkts = []
    for k in range(600):
        body = bytearray(rng.choice(b"abcdefghijklmnop ") for _ in range(rng.choice([0, 5, 60, 300, 1400])))
        for _ in range(rng.randint(0, 3)):
            if len(body) > 8:
                t = rng.choice(tokens)
                at = rng.randint(0, max(0, len(body) - len(t)))
                body[at:at + len(t)] = t[: len(body) - at]
        pkts.append(bytes(body))
    window = [(0, 40) if i % 3 == 0 else (10, 700) if i % 3 == 1 else None for i in range(len(tokens))]
    if kind == "all_windowed":
        window = [w or (0, 1399) for w in window]
    nocase = [i % 4 == 0 for i in range(len(tokens))]
    want_counts, want, verdicts = check_forms(engines, tokens, *csr(pkts), nocase, window, label=kind)
    assert sum(want_counts) > 100
    union, perpat = engines
    # the savefile forms and the frame stream
    path = str(tmp_path / "w.pcap")
    frames = [udp_frame(p) for p in pkts]
    write_pcap(path, frames)
    for m in (union, perpat):
        assert m.count_pcap(path) == want_counts
        assert m.count_pcap_streamed(path) == want_counts
        with m.stream("udp", batch_bytes=1 << 16) as st:
            for f in frames:
                st.push(f)
            assert st.flush() == want_counts
    got = union.find_pcap(path)
    assert np.array_equal(got[ORDER].astype(kmp.MATCH_DTYPE), want)
    assert np.array_equal(union.select_pcap(path), verdicts)


@pytest.mark.gpu
@pytest.mark.parametrize("pcap", PCAPS)
@pytest.mark.parametrize("proto", ["udp", "tcp"])
def test_bundled_savefiles_and_command_lines(engines, oracle, pcap, proto, tmp_path):
    union, perpat = engines
    path = os.path.join(DATA, pcap + ".pcap")
    tokens = oracle.load_patterns(STRINGS)
    data, offsets, _ = oracle.load_pcap_csr(path, proto)
    lo, hi = 3, 150
    frames = pcap_frames(path)
    accepted = [i for i, f in enumerate(frames) if oracle.extract(f, proto) is not None]
    for nocase in (False, True):
        ic = ["-i"] if nocase else []
        want_counts, want, verdicts = expected(tokens, data, offsets, nocase, (lo, hi))
        for m in (union, perpat):
            m.set_patterns(tokens, nocase, (lo, hi))
            assert m.window == [(lo, hi)] * len(tokens)
            assert m.count_pcap(path, proto) == want_counts
            assert m.count_pcap_streamed(path, proto) == want_counts
        got = union.find_pcap(path, proto)
        assert np.array_equal(got[ORDER].astype(kmp.MATCH_DTYPE), want)
        assert np.array_equal(union.select_pcap(path, proto), verdicts)
        # kmp_match -w: the report of the windowed counts (-i and -w in either order)
        report = oracle.format_report(tokens, want_counts)
        for opts in (ic + ["-w", "%d:%d" % (lo, hi)], ["-w", "%d:%d" % (lo, hi)] + ic):
            r = subprocess.run([MATCH, *opts, path, STRINGS, proto], capture_output=True)
            assert r.returncode == 0, r.stderr
            lines = r.stdout.splitlines(keepends=True)
            assert lines[-1].startswith(b"Elapsed time = ") and b"".join(lines[:-1]) == report, opts
        # kmp_find -w: the unwindowed lines whose offset lies in the window
        full = subprocess.run([FIND, *ic, path, STRINGS, proto], capture_output=True)
        r = subprocess.run([FIND, *ic, "-w", "%d:%d" % (lo, hi), path, STRINGS, proto], capture_output=True)
        assert full.returncode == 0 and r.returncode == 0, r.stderr
        keep = [ln for ln in full.stdout.decode("latin-1").splitlines() if lo <= int(ln.split(" ")[1]) <= hi]
        assert r.stdout.decode("latin-1").splitlines() == keep
        assert len(keep) == len(want)
        # kmp_select -w: the written frames are the selected ones; kmp_match -w counts the same in them
        out = str(tmp_path / ("sel%d.pcap" % nocase))
        r = subprocess.run([SELECT, "-w", "%d:%d" % (lo, hi), *ic, path, STRINGS, out, proto], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        assert r.stdout == "%d of %d packets written to %s\n" % (int(verdicts.sum()), len(verdicts), out)
        if verdicts.any():
            r = subprocess.run([MATCH, *ic, "-w", "%d:%d" % (lo, hi), out, STRINGS, proto], capture_output=True)
            assert r.returncode == 0 and b"".join(r.stdout.splitlines(keepends=True)[:-1]) == report


@pytest.mark.gpu
def test_host_find_forms_overflow_and_rematch(monkeypatch, tmp_path):
    monkeypatch.setenv("KMPB_CHUNK_MB", "1")
    packets = [b"a" * 8192] * 640  # 4096 windowed records a packet: every chunk overflows its slot's buffer
    data, offsets = csr(packets)
    want_counts, want, _ = expected([b"a"], data, offsets, False, (0, 4095))
    assert len(want) == 640 * 4096
    path = str(tmp_path / "dense.pcap")
    write_pcap(path, [udp_frame(p) for p in packets])
    with kmp.Matcher(0) as m:
        for win in ((0, 4095), [(0, 4095), None]):
            pats = [b"a"] if isinstance(win, tuple) else [b"a", b"aa"]
            wc, w, _ = expected(pats, data, offsets, False, win)
            m.set_patterns(pats, window=win)
            assert m.count_host(data, offsets) == wc
            assert np.array_equal(m.find_host(data, offsets), w)
            assert np.array_equal(m.find_pcap(path)[ORDER].astype(kmp.MATCH_DTYPE), w)
            assert m.count_pcap_streamed(path) == wc


@pytest.mark.gpu
def test_device_batch_past_4GiB():
    import torch

    L = 4096
    n = (9 << 29) // L  # 4.5 GiB of 4096-byte packets
    try:
        d_bytes = torch.full((n * L + 64,), ord("x"), dtype=torch.uint8, device="cuda:0")
    except RuntimeError:
        pytest.skip("not enough device memory")
    d_off = torch.arange(0, n + 1, dtype=torch.int64, device="cuda:0") * L
    k32 = (1 << 32) // L
    plants = [k32 - 2, k32 - 1, k32, k32 + 1, n - 1]  # packets that start just below and at / above 2^32
    for k in plants:
        d_bytes[k * L: k * L + 4] = torch.tensor(list(b"GET "), dtype=torch.uint8)
        d_bytes[k * L + 9: k * L + 11] = torch.tensor(list(b"QZ"), dtype=torch.uint8)
    d_bytes[k32 * L - 2: k32 * L] = torch.tensor(list(b"QZ"), dtype=torch.uint8)  # ends packet k32 - 1, offset 4094
    pats = [b"GET ", b"QZ", b"QZ", b"xQ"]
    win = [(0, 0), (9, 9), None, (4093, 4095)]
    want_counts = [len(plants), len(plants), len(plants) + 1, 1]  # "xQ" of every plant lies at offset 8: outside
    want = sorted([(k, 0, 0) for k in plants] + [(k, 9, 1) for k in plants] + [(k, 9, 2) for k in plants] +
                  [(k32 - 1, 4094, 2), (k32 - 1, 4093, 3)])
    span = (0, n * L)
    for engine in ("union", "perpat"):
        with kmp.Matcher(0, engine=engine) as m:
            m.set_patterns(pats, window=win)
            d_counts = torch.zeros(len(pats), dtype=torch.int64, device="cuda:0")
            m.count_device(d_bytes.data_ptr(), d_off.data_ptr(), n, d_counts.data_ptr(), span=span)
            torch.cuda.synchronize()
            assert d_counts.cpu().tolist() == want_counts, engine
            if engine == "perpat":
                continue
            cap = len(want) + 4
            d_out = torch.zeros(cap * 16, dtype=torch.uint8, device="cuda:0")
            d_n = torch.zeros(1, dtype=torch.int64, device="cuda:0")
            m.find_device(d_bytes.data_ptr(), d_off.data_ptr(), n, d_out.data_ptr(), cap, d_n.data_ptr(), span, sorted=True)
            torch.cuda.synchronize()
            rec = d_out.cpu().numpy()[: 16 * int(d_n.item())].view(kmp.MATCH_DTYPE)
            assert as_tuples(rec) == want
            d_flags = torch.zeros(n, dtype=torch.uint8, device="cuda:0")
            d_index = torch.zeros(n, dtype=torch.int64, device="cuda:0")
            d_sel = torch.zeros(1, dtype=torch.int64, device="cuda:0")
            m.select_device(d_bytes.data_ptr(), d_off.data_ptr(), n, d_flags.data_ptr(), span, d_index.data_ptr(),
                            d_sel.data_ptr())
            torch.cuda.synchronize()
            assert d_index[: int(d_sel.item())].cpu().tolist() == plants
            kmp.matcher.check(kmp.lib().kmpb_check_device_errors(m.handle))
    del d_bytes, d_off
    torch.cuda.empty_cache()


@pytest.mark.gpu
def test_interleaved_with_calls_in_flight_and_a_frame_stream():
    import torch

    tokens = kmp.load_patterns(STRINGS)
    rng = random.Random(3)
    pkts = [bytes(rng.choice(b"abcdefgh tp/") for _ in range(rng.choice([10, 200, 1400]))) + rng.choice(tokens) for _ in range(3000)]
    data, offsets = csr(pkts)
    window = [(0, 300) if i % 2 else None for i in range(len(tokens))]
    want_counts, want, verdicts = expected(tokens, data, offsets, False, window)
    with kmp.Matcher(0) as m:
        m.set_patterns(tokens, window=window)
        batch = DeviceBatch(data, offsets)
        d_counts = torch.zeros(len(tokens), dtype=torch.int64, device="cuda:0")
        side = torch.cuda.Stream()
        for _ in range(4):  # device calls in flight on a side stream, host forms behind them
            m.count_device(batch.d_bytes.data_ptr(), batch.d_off.data_ptr(), len(pkts), d_counts.data_ptr(),
                           span=(0, int(offsets[-1])), stream=side.cuda_stream)
        assert np.array_equal(m.find_host(data, offsets), want)
        assert m.count_host(data, offsets) == want_counts
        torch.cuda.synchronize()
        assert d_counts.cpu().tolist() == [4 * c for c in want_counts]
        frames = [udp_frame(p) for p in pkts]
        with m.stream("udp", batch_bytes=1 << 17) as st:
            for f in frames[:1500]:
                st.push(f)
            with pytest.raises(kmp.KmpbError):
                m.set_patterns(tokens, window=(0, 5))  # the open stream owns the context
            for f in frames[1500:]:
                st.push(f)
            assert st.flush() == want_counts
        flags, counts = m.select_host(data, offsets)
        assert np.array_equal(flags, verdicts) and counts == want_counts


@pytest.mark.gpu
def test_randomised_mixed_sets(engines):
    rng = random.Random(2026)
    alpha = b"aAbBcz\0"
    for trial in range(300):
        pats = [bytes(rng.choice(alpha[:-1]) for _ in range(rng.choice([1, 1, 2, 3, 4, 9]))) for _ in range(rng.randint(1, 7))]
        if len(pats) > 1 and trial % 3 == 0:
            pats.append(pats[0])
        nocase = [rng.random() < 0.3 for _ in pats]
        window = []
        for _ in pats:
            lo = rng.choice([0, 0, 1, 3, 40, 130])
            window.append(None if rng.random() < 0.35 else (lo, lo + rng.choice([0, 1, 5, 100, 2000])))
        pkts = [bytes(rng.choice(alpha) for _ in range(rng.choice([0, 1, 4, 30, 200, 1500]))) for _ in range(rng.randint(1, 12))]
        check_forms(engines, pats, *csr(pkts), nocase, window, label=trial,
                    forms=HOST_FORMS + DEVICE_FORMS if trial % 25 == 0 else HOST_FORMS)
