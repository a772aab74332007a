"""Position windows at scale: windowed sets large enough that the window kernel (csrc/cuda/window.cu) keeps its
counters or its probe tables in global memory, walks runs of thousands of one-byte patterns, and compares long
patterns at tile edges -- through both engines and every form, against an exact reference.

The reference is the numpy one of tests/kmpb_reference.py, which costs about one table lookup per text byte and
distinct (flag, length), not patterns x bytes.  The CPU tests check it against the naive finder and the
reference-finder answers of the same module.

The kernel's two placement decisions (`kmpb_launch_window`): the counters go to shared memory for at most 4096
distinct windowed patterns (8 * n_win <= 32768), the probe tables for at most 16384 words (4 * wvtab_words <= 65536).
tests/c/window_geometry.c prints what automaton.c builds for a set, and the CPU tests assert which side of each
condition every case lies on, so that a change to the table builder that moves a case off its path fails here
without a GPU."""
import functools
import os
import random
import subprocess

import numpy as np
import pytest

from conftest import ROOT
from kmpb_harness import check_forms, engines, udp_frame, write_pcap  # noqa: F401
from kmpb_reference import ORDER, csr, expected, firsts, fold, naive, normalise, reference

import multithreading_string_matching_b200 as kmp

HOSTC = os.path.join(ROOT, "multithreading_string_matching_b200", "csrc", "host")
ANY = 0xFFFFFFFF
COUNTS_SMEM_MAX = 4096  # window.cu: distinct windowed patterns whose 64-bit counters stay in shared memory
VTAB_SMEM_MAX = 16384   # window.cu: words of probe tables that stay in shared memory
TILE = 1024             # window.cu WN_TILE: start offsets per tile
LOWER = b"abcdefghijklmnopqrstuvwxyz"
MIXED = LOWER + LOWER.upper() + b"0123456789"


# ---- the tables' geometry -------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def geometry(tmp_path_factory):
    """set -> (n_pat, n_uniq, n_union, wvtab_words) from automaton.c (tests/c/window_geometry.c)"""
    d = tmp_path_factory.mktemp("window_geometry")
    exe = str(d / "window_geometry")
    subprocess.run(["/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc", "-O1", "-I" + os.path.join(ROOT, "include"),
                    "-I" + HOSTC, os.path.join(ROOT, "tests", "c", "window_geometry.c"), os.path.join(HOSTC, "automaton.c"),
                    os.path.join(HOSTC, "errors.c"), "-o", exe], check=True)

    def run(patterns, nocase, window):
        patterns, nocase, window = normalise(patterns, nocase, window)
        path = str(d / "set.txt")
        with open(path, "w") as f:
            for p, nc, w in zip(patterns, nocase, window):
                lo, hi = w if w is not None else (0, ANY)
                f.write("%d %d %d %s\n" % (int(nc), lo, hi, p.hex()))
        r = subprocess.run([exe, path], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        return tuple(int(x) for x in r.stdout.split())

    return run


def paths(g):
    """(counters in shared memory, probe tables in shared memory) of window.cu for a set's geometry"""
    n_pat, n_uniq, n_union, wvtab_words = g
    return n_uniq - n_union <= COUNTS_SMEM_MAX, wvtab_words <= VTAB_SMEM_MAX


def longest_run(patterns, nocase, window):
    """the most distinct windowed one-byte patterns of one byte and flag (the kernel walks down such a run)"""
    patterns, nocase, window = normalise(patterns, nocase, window)
    runs = {}
    for p, nc, w in {(fold(p) if nc else p, nc, w) for p, nc, w in zip(patterns, nocase, window)}:
        if len(p) == 1 and w is not None:
            runs[(p, nc)] = runs.get((p, nc), 0) + 1
    return max(runs.values(), default=0)


def distinct_windowed(patterns, nocase, window):
    patterns, nocase, window = normalise(patterns, nocase, window)
    return len({(fold(p) if nc else p, nc, w) for p, nc, w in zip(patterns, nocase, window) if w is not None})


# ---- the sets and their packets -------------------------------------------------------------------------------------

def narrow_window(rng, lo_max=1500):
    lo = rng.randrange(0, lo_max)
    return (lo, lo + rng.choice([0, 1, 3, 40, 300]))


def boundary_sequence():
    """a seeded sequence of case-sensitive windowed patterns of 3-12 bytes; its prefixes grow the window tables"""
    rng = random.Random(71)
    pats = [bytes(rng.choice(LOWER) for _ in range(rng.randint(3, 12))) for _ in range(1400)]
    return pats, [narrow_window(rng, 600) for _ in pats]


@functools.lru_cache(maxsize=None)
def _boundary_n(run):
    """the longest prefix of boundary_sequence whose window tables fit in shared memory (binary search: the tables
    only grow with the set)"""
    pats, win = boundary_sequence()
    lo, hi = 1, len(pats)
    assert paths(run(pats[:lo], False, win[:lo]))[1] and not paths(run(pats, False, win))[1]
    while hi - lo > 1:
        mid = (lo + hi) // 2
        if paths(run(pats[:mid], False, win[:mid]))[1]:
            lo = mid
        else:
            hi = mid
    return lo


def boundary_sets(geometry):
    pats, win = boundary_sequence()
    n = _boundary_n(geometry)
    return [(pats[:n], False, win[:n]), (pats[:n + 1], False, win[:n + 1])]


def nocase_tails_set():
    """about 200 nocase windowed patterns of 2-40 bytes and 40 case-sensitive ones"""
    rng = random.Random(72)
    pats = [bytes(rng.choice(MIXED) for _ in range(rng.randint(2, 40))) for _ in range(240)]
    nocase = [i < 200 for i in range(240)]
    return pats, nocase, [narrow_window(rng) for _ in pats]


def runs_set(n_distinct):
    """n_distinct distinct windowed patterns, most of them long runs of one-byte patterns (one byte and flag, distinct
    narrow windows): case-sensitive and nocase runs of `a`, a case-sensitive run of `A`, a nocase run of `7`, and a
    few two-byte patterns; shuffled, so that file order is not id order, with duplicates of some of them"""
    rng = random.Random(73)
    pats, nocase, window = [], [], []
    two = [(b"ab", False), (b"aB", True), (b"a7", False), (b"7a", True), (b"Aa", False)]
    for k, (p, nc) in enumerate(two):
        pats.append(p)
        nocase.append(nc)
        window.append((k * 13, k * 13 + 900))
    runs = [(b"a", False, 1500), (b"a", True, 1400), (b"A", False, 600), (b"7", True, n_distinct - 3500 - len(two))]
    for byte, nc, length in runs:
        for k in range(length):
            lo = (k * 37) % 2500  # distinct for every k < 2500
            pats.append(byte)
            nocase.append(nc)
            window.append((lo, lo + k % 3))
    order = list(range(len(pats)))
    rng.shuffle(order)
    order += [order[k] for k in (3, 500, 2000)]
    return [pats[i] for i in order], [nocase[i] for i in order], [window[i] for i in order]


def big_windowed_set():
    """about 5000 windowed patterns of 2-99 bytes, mixed flags; the same bytes under several windows, and duplicates of
    one (bytes, flag, window) far apart in file order"""
    rng = random.Random(74)
    pats, nocase, window = [], [], []
    for _ in range(4700):
        m = rng.choice([2, 3, 4, 5, 6, 7, 8, 9, 12, 16, 33, 64, 99])
        pats.append(bytes(rng.choice(MIXED) for _ in range(m)))
        nocase.append(rng.random() < 0.3)
        window.append(narrow_window(rng))
    for k in range(0, 300, 3):  # the same bytes and flag under other windows
        pats.append(pats[k])
        nocase.append(nocase[k])
        window.append(narrow_window(rng))
    for k in (7, 1234, 2500):  # duplicates, far from their first index
        pats.insert(len(pats) // 2 + k, pats[k])
        nocase.insert(len(nocase) // 2 + k, nocase[k])
        window.insert(len(window) // 2 + k, window[k])
        pats.append(pats[k])
        nocase.append(nocase[k])
        window.append(window[k])
    return pats, nocase, window


def mixed_scale_set():
    """more than 4096 unwindowed and more than 4096 windowed distinct patterns, the windowed ones the same bytes as
    unwindowed ones"""
    rng = random.Random(75)
    alpha = b"abcdefghijklmnop"
    pool = sorted({bytes(rng.choice(alpha) for _ in range(rng.randint(3, 12))) for _ in range(4400)})
    pats, nocase, window = [], [], []
    for p in pool:
        nc = rng.random() < 0.25
        pats += [p, p]
        nocase += [nc, nc if rng.random() < 0.8 else not nc]
        window += [None, narrow_window(rng, 1200)]
    order = list(range(len(pats)))
    rng.shuffle(order)
    return [pats[i] for i in order], [nocase[i] for i in order], [window[i] for i in order]


def tile_set(decoys=0):
    """windowed patterns of 9, 33, 64 and 99 bytes, case-sensitive and nocase, with windows around the tile edges
    and a reach max(hi + len) that is not a multiple of 16; `decoys` more windowed patterns that never occur"""
    rng = random.Random(76)
    window = [(1000, 4101), (1023, 4096), (0, 2047), (1024, 3071), (2047, 4100), (1023, 1024), (2047, 4101), (3071, 4096)]
    pats, nocase = [], []
    for m in (9, 33, 64, 99):
        for nc in (False, True):
            pats.append(bytes(rng.choice(b"abcdefgh") for _ in range(m)))
            nocase.append(nc)
    for _ in range(decoys):
        pats.append(bytes(rng.choice(b"qrstuvwxyz") for _ in range(rng.randint(3, 12))))
        nocase.append(rng.random() < 0.2)
        window.append((rng.randrange(1000, 4000), 4101))
    return pats, nocase, window


EDGES = [e for t in range(1, 5) for e in (t * TILE - 1, t * TILE)]  # the last and first start of tiles 0..3


def tile_packets():
    """every tile-set pattern planted at every tile edge, in packets that start at every residue mod 16; a NUL at the
    match's last byte, one byte past it, in the lookahead of the match's tile, or none"""
    rng = random.Random(77)
    pats, nocase, _ = tile_set()
    pkts, cur, combos = [], 0, []
    for pi in range(len(pats)):
        for ei, e in enumerate(EDGES):
            for r in range(16):
                combos.append((pi, ei, e, r))
    rng.shuffle(combos)
    for k, (pi, ei, e, r) in enumerate(combos):
        assert cur % 16 == r or k == 0
        p, m = pats[pi], len(pats[pi])
        body = bytearray(rng.choice(b"abcdefgh") for _ in range(e + m + rng.choice([0, 1, 7, 150])))
        body[e: e + m] = bytes(c ^ 0x20 if nocase[pi] and rng.random() < 0.5 else c for c in p)
        variant = (r + ei) % 4
        if variant == 1:
            body[e + m - 1] = 0
        elif variant == 2 and len(body) > e + m:
            body[e + m] = 0
        elif variant == 3:
            at = (e // TILE) * TILE + TILE + 127  # the last lookahead byte of the match's tile
            if at < len(body):
                body[at] = 0
        nxt = combos[k + 1][3] if k + 1 < len(combos) else 0
        body += bytes(rng.choice(b"abcdefgh") for _ in range((nxt - (cur + len(body))) % 16))
        pkts.append(bytes(body))
        cur += len(body)
    return pkts


def planted(seed, patterns, nocase, window, n_packets, sizes, alpha, plants=24, nul=0.05):
    """packets of random bytes from alpha with patterns written in: most at offsets inside their window or one off
    its edges, nocase ones in random case; a few packets with a NUL"""
    patterns, nocase, window = normalise(patterns, nocase, window)
    rng = random.Random(seed)
    npr = np.random.default_rng(seed)
    abytes = np.frombuffer(alpha, dtype=np.uint8)
    pkts = []
    for _ in range(n_packets):
        body = bytearray(npr.choice(abytes, rng.choice(sizes)).tobytes())
        for _ in range(rng.randint(0, plants)):
            i = rng.randrange(len(patterns))
            p, w = patterns[i], window[i]
            if w is None:
                at = rng.randint(0, max(0, len(body) - len(p)))
            else:
                at = rng.choice([w[0], w[1], w[0] - 1, w[1] + 1, rng.randint(w[0], w[1])])
            if at < 0 or at + len(p) > len(body):
                continue
            body[at: at + len(p)] = bytes(c ^ 0x20 if nocase[i] and chr(c).isalpha() and rng.random() < 0.5 else c for c in p)
        if body and rng.random() < nul:
            body[rng.randrange(len(body))] = 0
        pkts.append(bytes(body))
    return pkts


# ---- CPU: the reference ---------------------------------------------------------------------------------------------

def test_reference_against_the_naive_finder():
    rng = random.Random(81)
    alpha = b"aAbz\0"
    for trial in range(300):
        pats = [bytes(rng.choice(alpha[:-1]) for _ in range(rng.randint(1, 5))) for _ in range(rng.randint(1, 9))]
        nocase = [rng.random() < 0.4 for _ in pats]
        window = [None if rng.random() < 0.3 else (lambda lo: (lo, lo + rng.randint(0, 12)))(rng.randint(0, 10)) for _ in pats]
        if trial % 2:  # duplicates, the same bytes under another window, and the same bytes in another flag
            k = rng.randrange(len(pats))
            pats += [pats[k], pats[k], pats[k].upper()]
            nocase += [nocase[k], nocase[k], not nocase[k]]
            window += [window[k], (0, rng.randint(0, 20)), window[k]]
        pkts = [bytes(rng.choice(alpha) for _ in range(rng.randint(0, 30))) for _ in range(rng.randint(0, 6))]
        data, offsets = csr(pkts)
        counts, rec, verdicts = reference(pats, nocase, window, data, offsets)
        want = naive(pkts, pats, nocase, window)
        first = firsts(pats, nocase, window)
        assert list(zip(rec["packet"].tolist(), rec["offset"].tolist(), rec["pattern"].tolist())) == want, trial
        assert verdicts.tolist() == [any(r[0] == k for r in want) for k in range(len(pkts))], trial
        assert counts == [sum(1 for r in want if r[2] == first[i]) for i in range(len(pats))], trial


def test_reference_against_the_reference_finder():
    rng = random.Random(82)
    for trial in range(6):
        pats = [bytes(rng.choice(b"abcdAB") for _ in range(rng.choice([1, 2, 3, 5, 9, 14, 40]))) for _ in range(300)]
        nocase = [rng.random() < 0.3 for _ in pats]
        window = [None if trial % 2 and rng.random() < 0.4 else narrow_window(rng, 400) for _ in pats]
        pkts = planted(trial, pats, nocase, window, 120, [0, 30, 400, 1500], b"abcdAB", plants=6, nul=0.3)
        data, offsets = csr(pkts)
        got = reference(pats, nocase, window, data, offsets)
        want = expected(pats, data, offsets, nocase, window)
        assert got[0] == want[0] and np.array_equal(got[1], want[1]) and np.array_equal(got[2], want[2]), trial
        assert len(want[1]) > 1000


# ---- CPU: which path each case takes --------------------------------------------------------------------------------

def test_case_paths(geometry):
    # 1: the last set whose tables fit in shared memory and the first that does not, counters shared
    below, above = (geometry(*s) for s in boundary_sets(geometry))
    assert paths(below) == (True, True) and paths(above) == (True, False)
    assert above[0] == below[0] + 1 and below[3] <= VTAB_SMEM_MAX < above[3]
    # 2: tables global with nocase patterns of more than 8 bytes (their tail masks are read from global memory)
    pats, nocase, window = nocase_tails_set()
    assert paths(geometry(pats, nocase, window)) == (True, False)
    assert any(nc and len(p) > 8 for p, nc in zip(pats, nocase))
    # 3: 4096 and 4097 distinct windowed patterns in runs of up to 1500 one-byte patterns, tables shared
    for n, counts_shared in ((4096, True), (4097, False)):
        s = runs_set(n)
        g = geometry(*s)
        assert g[2] == 0 and g[1] == n == distinct_windowed(*s) and paths(g) == (counts_shared, True)
        assert longest_run(*s) == 1500
    # 4 and 6: about 5000 windowed patterns, all windowed: counters and tables global, more than 256 patterns expanded
    s = big_windowed_set()
    g = geometry(*s)
    assert g[2] == 0 and g[1] == distinct_windowed(*s) < len(s[0]) and paths(g) == (False, False) and g[0] > 256
    # 5: more than 4096 distinct patterns of each kind: the window kernel's counters global
    s = mixed_scale_set()
    g = geometry(*s)
    assert g[2] > COUNTS_SMEM_MAX and g[1] - g[2] == distinct_windowed(*s) > COUNTS_SMEM_MAX and not paths(g)[0]
    # 7: the tile set alone (tables shared) and padded past the table boundary (tables global); its reach
    for decoys, tables_shared in ((0, True), (900, False)):
        s = tile_set(decoys)
        assert paths(geometry(*s)) == (True, tables_shared)
        reach = max(w[1] + len(p) for p, w in zip(s[0], s[2]))
        assert reach % 16 and reach > EDGES[-1] + 99


def test_tile_packets_cover_every_lead():
    pkts = tile_packets()
    _, offsets = csr(pkts)
    assert len(pkts) == 8 * len(EDGES) * 16
    assert set((offsets[:-1] % 16).tolist()) == set(range(16))


# ---- GPU ------------------------------------------------------------------------------------------------------------

def run_case(engines, s, pkts, label):
    data, offsets = csr(pkts)
    answers = reference(*s, data, offsets)
    assert sum(answers[0]) > 0, label
    return check_forms(engines, s[0], data, offsets, *s[1:], label=label, answers=answers)


@pytest.mark.gpu
def test_table_boundary(engines, geometry):
    for k, s in enumerate(boundary_sets(geometry)):
        run_case(engines, s, planted(10 + k, *s, 300, [0, 40, 300, 1200, 2500], LOWER), "boundary %d" % k)


@pytest.mark.gpu
def test_global_tables_with_nocase_tail_masks(engines):
    s = nocase_tails_set()
    run_case(engines, s, planted(12, *s, 300, [0, 60, 700, 2000], MIXED), "nocase tails")


@pytest.mark.gpu
@pytest.mark.parametrize("n", [4096, 4097])
def test_runs_of_one_byte_patterns_at_the_counter_boundary(engines, n):
    s = runs_set(n)
    run_case(engines, s, planted(13, *s, 200, [1, 100, 1500, 2600], b"aA7bx", plants=0), "runs %d" % n)


@pytest.mark.gpu
def test_all_windowed_global_counters_and_tables(engines):
    s = big_windowed_set()
    run_case(engines, s, planted(14, *s, 300, [0, 50, 600, 1800, 3000], MIXED), "all windowed")


@pytest.mark.gpu
def test_mixed_at_scale(engines):
    s = mixed_scale_set()
    want_counts, want, _ = run_case(engines, s, planted(15, *s, 300, [0, 50, 600, 1800], b"abcdefghijklmnop"), "mixed")
    # one text occurrence of shared bytes is a record of each kind
    pats, _, window = s
    kinds = {(int(r["packet"]), int(r["offset"]), window[int(r["pattern"])] is None) for r in want}
    both = {(k, o) for k, o, unw in kinds if unw} & {(k, o) for k, o, unw in kinds if not unw}
    assert len(both) > 100


@pytest.mark.gpu
@pytest.mark.parametrize("decoys", [0, 900])
def test_tile_edges_with_long_patterns(engines, decoys):
    s = tile_set(decoys)
    run_case(engines, s, tile_packets(), "tiles %d" % decoys)


@pytest.mark.gpu
@pytest.mark.parametrize("which", ["all_windowed", "mixed"])
def test_chunked_host_and_savefile_forms(monkeypatch, which, tmp_path):
    monkeypatch.setenv("KMPB_CHUNK_MB", "1")
    s = big_windowed_set() if which == "all_windowed" else mixed_scale_set()
    alpha = MIXED if which == "all_windowed" else b"abcdefghijklmnop"
    pkts = planted(16, *s, 2200, [0, 600, 1800, 3000, 5000, 8000], alpha)
    data, offsets = csr(pkts)
    assert int(offsets[-1]) >= 5 << 20  # at least 5 chunks: every stream slot retires a chunk, one of them twice
    want_counts, want, verdicts = reference(*s, data, offsets)
    assert len(want) > 1000
    path = str(tmp_path / "w.pcap")
    frames = [udp_frame(p) for p in pkts]
    write_pcap(path, frames)
    with kmp.Matcher(0, engine="union") as union, kmp.Matcher(0, engine="perpat") as perpat:
        for m in (union, perpat):
            m.set_patterns(*s)
            assert m.count_host(data, offsets) == want_counts, (which, m is union)
            assert m.count_pcap(path) == want_counts, (which, m is union)
            assert m.count_pcap_streamed(path) == want_counts, (which, m is union)
            with m.stream("udp", batch_bytes=1 << 20) as st:
                for f in frames:
                    st.push(f)
                assert st.flush() == want_counts, (which, m is union)
        assert np.array_equal(union.find_host(data, offsets), want)
        assert np.array_equal(union.find_pcap(path)[ORDER].astype(kmp.MATCH_DTYPE), want)
        flags, counts = union.select_host(data, offsets)
        assert np.array_equal(flags, verdicts) and counts == want_counts
        assert np.array_equal(union.select_pcap(path), verdicts)
        kmp.matcher.check(kmp.lib().kmpb_check_device_errors(union.handle))
