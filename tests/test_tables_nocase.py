"""Case-insensitive patterns without a GPU: the host tables (tests/c/test_tables_nocase.c against csrc/host/automaton.c),
the usage text of `kmp_match -i` / `kmp_find -i`, and the derivation of the expected answers (tests/kmpb_reference.py
`expected`: a nocase pattern's matches are the case-sensitive matches of the folded pattern in the folded text, the
oracle's counts of each flag group alongside), checked against a naive finder."""
import os
import random
import subprocess

import numpy as np
import pytest

from conftest import ROOT
from kmpb_harness import BIN
from kmpb_reference import csr, expected, firsts, fold, naive

HOSTC = os.path.join(ROOT, "multithreading_string_matching_b200", "csrc", "host")


def test_host_tables_nocase_selfcheck(tmp_path):
    """All-zero flags build the tables of kmpb_tables_build word for word; on random mixed sets every case variant passes
    the filter and the gate and finds its record, the masks accept exactly the case variants, and the probe tables and
    the merged DFA count what a naive folded counter counts."""
    exe = str(tmp_path / "test_tables_nocase")
    subprocess.run(["/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc", "-O1", "-g", "-I" + os.path.join(ROOT, "include"),
                    "-I" + HOSTC, os.path.join(ROOT, "tests", "c", "test_tables_nocase.c"), os.path.join(HOSTC, "automaton.c"),
                    os.path.join(HOSTC, "errors.c"), "-o", exe], check=True)
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr


@pytest.mark.parametrize("prog,usage", [("kmp_match", "USAGE: ./kmp_match <file.pcap> <string.txt> [tcp/udp]\n"),
                                        ("kmp_find", "USAGE: ./kmp_find <file.pcap> <string.txt> [tcp/udp]\n")])
def test_dash_i_with_missing_arguments_prints_the_usage(prog, usage):
    exe = os.path.join(BIN, prog)
    for argv in (["-i"], ["-i", "a.pcap"]):
        r = subprocess.run([exe, *argv], capture_output=True, text=True)
        assert r.returncode == 1 and r.stdout == usage, (argv, r.stdout, r.stderr)
    r = subprocess.run([exe, "-i", "a", "b", "icmp"], capture_output=True, text=True)
    assert r.returncode == 1 and r.stdout == usage.replace("USAGE: ", "USAGE "), r.stdout


def test_fold_is_ascii_letters_only():
    assert fold(bytes(range(256))) == bytes(c + 32 if 0x41 <= c <= 0x5A else c for c in range(256))
    assert fold(b"@[\\]^_\x7f\xc1\xdf`{|}~") == b"@[\\]^_\x7f\xc1\xdf`{|}~"


def test_expected_answers_against_a_naive_finder(oracle):
    rng = random.Random(7)
    alpha = b"aAbBzZ@`[{^~_\x7f\xc1\xe1\0"
    for trial in range(150):
        pats = [bytes(rng.choice(alpha[:-1]) for _ in range(rng.randint(1, 5))) for _ in range(rng.randint(1, 8))]
        if trial % 3 == 0 and len(pats) > 1:  # an earlier token in another case
            pats.append(pats[0].swapcase())
        nocase = [rng.random() < 0.5 for _ in pats]
        pkts = [bytes(rng.choice(alpha) for _ in range(rng.randint(0, 40))) for _ in range(rng.randint(1, 6))]
        data, offsets = csr(pkts)
        counts, rec, _ = expected(pats, data, offsets, nocase, oracle=oracle)
        want = naive(pkts, pats, nocase)
        assert list(zip(rec["packet"].tolist(), rec["offset"].tolist(), rec["pattern"].tolist())) == want, trial
        first = firsts(pats, nocase)
        hist = np.bincount(rec["pattern"].astype(np.int64), minlength=len(pats))
        assert counts == [int(hist[first[i]]) for i in range(len(pats))], trial
