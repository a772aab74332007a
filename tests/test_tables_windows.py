"""Position windows without a GPU: the host tables (tests/c/test_tables_windows.c against csrc/host/automaton.c), the
`-w` option of the three command lines (malformed values, exit codes, unchanged usage texts), Matcher's argument
checks, and the derivation of the expected answers (tests/kmpb_reference.py `expected`) checked against a naive
finder."""
import hashlib
import json
import os
import random
import subprocess

import pytest

from conftest import ROOT
from kmpb_harness import BIN
from kmpb_reference import csr, expected, firsts, naive

import multithreading_string_matching_b200 as kmp

HOSTC = os.path.join(ROOT, "multithreading_string_matching_b200", "csrc", "host")


def test_host_tables_windows_selfcheck(tmp_path):
    exe = str(tmp_path / "test_tables_windows")
    subprocess.run(["/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc", "-O1", "-g", "-I" + os.path.join(ROOT, "include"),
                    "-I" + HOSTC, os.path.join(ROOT, "tests", "c", "test_tables_windows.c"), os.path.join(HOSTC, "automaton.c"),
                    os.path.join(HOSTC, "errors.c"), "-o", exe], check=True)
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr


@pytest.mark.parametrize("mode", ["0", "1", "2"])
@pytest.mark.parametrize("form", ["flags", "win"])
def test_tables_without_windows_are_those_built_before_windows(mode, form, tmp_path):
    """strings.txt without windows (kmpb_tables_build_flags, and kmpb_tables_build_win with every window {0,
    KMPB_WINDOW_ANY}) against hashes of the tables the library built before windows existed"""
    exe = str(tmp_path / "dump_tables")
    subprocess.run(["/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc", "-O1", "-fopenmp", "-I" + os.path.join(ROOT, "include"),
                    "-I" + HOSTC, os.path.join(ROOT, "tests", "c", "dump_tables.c"), os.path.join(HOSTC, "automaton.c"),
                    os.path.join(HOSTC, "errors.c"), os.path.join(HOSTC, "patterns.c"), "-o", exe], check=True)
    r = subprocess.run([exe, os.path.join(ROOT, "tests", "golden", "data", "strings.txt"), mode] + (["win"] if form == "win" else []),
                       capture_output=True, check=True)
    golden = json.load(open(os.path.join(ROOT, "tests", "golden", "tables_sha256.json")))
    assert hashlib.sha256(r.stdout).hexdigest() == golden[mode]


BAD = ["", "5", "5:", ":5", "5:3", "0:65536", "70000:70001", "a:3", "1:2x", "-1:3", "1:-3", " 1:3", "1: 3", "0x1:3", "1:3:5"]


@pytest.mark.parametrize("prog,extra", [("kmp_match", []), ("kmp_find", []), ("kmp_select", ["out.pcap"])])
def test_bad_window_is_an_error_before_any_device_work(prog, extra, tmp_path):
    exe = os.path.join(BIN, prog)
    for value in BAD:
        for argv in (["-w", value, "a.pcap", "s.txt", *extra], ["-i", "-w", value, "a.pcap", "s.txt", *extra]):
            r = subprocess.run([exe, *argv], capture_output=True, text=True, cwd=tmp_path)
            assert r.returncode == 1 and r.stdout == "" and r.stderr.startswith("error: bad window"), (argv, r.stdout, r.stderr)
    r = subprocess.run([exe, "-w"], capture_output=True, text=True, cwd=tmp_path)
    assert r.returncode == 1 and r.stderr.startswith("error: bad window")
    assert not os.path.exists(tmp_path / "out.pcap")


@pytest.mark.parametrize("prog,usage", [("kmp_match", "USAGE: ./kmp_match <file.pcap> <string.txt> [tcp/udp]\n"),
                                        ("kmp_find", "USAGE: ./kmp_find <file.pcap> <string.txt> [tcp/udp]\n"),
                                        ("kmp_select", "USAGE: ./kmp_select [-i] [-v] <file.pcap> <string.txt> <out.pcap> [tcp/udp]\n")])
def test_usage_texts_are_unchanged(prog, usage):
    exe = os.path.join(BIN, prog)
    for argv in ([], ["-w", "0:5"], ["-w", "0:5", "-i"], ["-i", "-w", "1:1", "a.pcap"]):
        r = subprocess.run([exe, *argv], capture_output=True, text=True)
        assert r.returncode == 1 and r.stdout == usage and r.stderr == "", (argv, r.stdout)


def test_matcher_window_argument_checks():
    m = kmp.Matcher.__new__(kmp.Matcher)  # argument checks run before any device call
    m._ctx = None
    with pytest.raises(ValueError):
        m.set_patterns([b"a", b"b", b"c"], window=[(0, 1), None])
    with pytest.raises(ValueError):
        m.set_patterns([b"a"], window=[(0, 1), (0, 2)])
    for bad in ((0, -1), (-1, 3), (0, 65536), (70000, 70001), [(0, 5), (0, 1 << 32)]):  # would wrap in uint32
        with pytest.raises(ValueError):
            m.set_patterns([b"a", b"b"], window=bad)


def test_expected_answers_against_a_naive_finder():
    rng = random.Random(9)
    alpha = b"aAbz\0"
    for trial in range(200):
        pats = [bytes(rng.choice(alpha[:-1]) for _ in range(rng.randint(1, 4))) for _ in range(rng.randint(1, 7))]
        if len(pats) > 1 and trial % 2:
            pats.append(pats[0])
        nocase = [rng.random() < 0.4 for _ in pats]
        window = [None if rng.random() < 0.3 else (lambda lo: (lo, lo + rng.randint(0, 12)))(rng.randint(0, 10)) for _ in pats]
        pkts = [bytes(rng.choice(alpha) for _ in range(rng.randint(0, 30))) for _ in range(rng.randint(1, 6))]
        data, offsets = csr(pkts)
        counts, rec, verdicts = expected(pats, data, offsets, nocase, window)
        want = naive(pkts, pats, nocase, window)
        assert list(zip(rec["packet"].tolist(), rec["offset"].tolist(), rec["pattern"].tolist())) == want, trial
        assert verdicts.tolist() == [any(r[0] == k for r in want) for k in range(len(pkts))]
        first = firsts(pats, nocase, window)
        assert counts == [sum(1 for r in want if r[2] == first[i]) for i in range(len(pats))]
