"""The union kernel's prefix gate (automaton.c build_gate, union_kernel.cu phase 1 of the resolve step): a start
position becomes a candidate only if the gate word of its first two bytes has the bit of its third byte set, and the
gate must let every true start through.  These tests put true starts where the gate is easiest to get wrong -- pattern
sets whose keys collide in the hash, short patterns that are prefixes of longer ones, starts in the last bytes of a
packet and of a work item, next to NULs and packet boundaries, at group offsets 29..31 (their key bytes lie in the
lookahead), bytes >= 0x80 -- and check both engines' counts against the oracle and every find form against the
reference finder (tests/c/kmp_find_ref.c).  A set with a one-byte pattern, or with very many keys, has no gate (the
resolve step re-runs the filter instead); those are checked the same way."""
import random

import numpy as np
import pytest

import multithreading_string_matching_b200 as kmp
from test_find import RefFinder, check_find, csr

GATE_MUL = 0x79B10000


def gate_geometry(patterns):
    """(words, shift) of the gate automaton.c builds for this set, or None when it builds none"""
    u = sorted(set(bytes(p) for p in patterns))
    keys = 256 * sum(len(p) == 1 for p in u) + len({p[:2] for p in u if len(p) >= 2})
    log_w = 5
    while (1 << log_w) < 1024 and (1 << log_w) < 16 * keys:
        log_w += 1
    shift = 32 - log_w
    g = [0] * (1 << log_w)
    for p in u:
        if len(p) == 1:
            for c in range(256):
                g[gate_slot(p[0] | c << 8, shift)] = 0xFFFFFFFF
        else:
            g[gate_slot(p[0] | p[1] << 8, shift)] |= 0xFFFFFFFF if len(p) == 2 else 0x80000000 >> (p[2] & 31)
    if not u or 8 * sum(bin(w).count("1") for w in g) > 32 * len(g):
        return None
    return 1 << log_w, shift


def gate_slot(key, shift):
    return ((key * GATE_MUL) & 0xFFFFFFFF) >> shift


def colliding_set(rng, alphabet):
    """patterns whose first two bytes share gate words: 80 random 3..12-byte patterns (enough keys for the largest
    table, 1024 words), then pairs of distinct keys with one slot, as 3-byte patterns whose third bytes are equal
    modulo 32 or equal, longer ones, and 2-byte patterns sharing their word with 3-byte ones"""
    pats = {bytes(rng.choice(alphabet) for _ in range(rng.randint(3, 12))) for _ in range(80)}
    by_slot, pairs = {}, 0
    keys = [a | b << 8 for a in alphabet for b in alphabet]
    rng.shuffle(keys)
    for k in keys:
        s = gate_slot(k, 22)
        k0 = by_slot.setdefault(s, k)
        if k0 != k and pairs < 8:
            a, b = bytes([k0 & 255, k0 >> 8]), bytes([k & 255, k >> 8])
            c = rng.choice(alphabet)
            pats |= {a + bytes([c]), b + bytes([c ^ 0x20 if c ^ 0x20 in alphabet else c]), b + bytes([c]) + b"q",
                     a + b"long" + a}
            if pairs % 2:
                pats.add(b)
            pairs += 1
    pats = sorted(pats)
    assert gate_geometry(pats) == (1024, 22) and pairs == 8
    return pats


def planted_packets(rng, pats, alphabet, n, size):
    """packets of random text with patterns planted at the places the gate has to get right"""
    pkts = []
    for i in range(n):
        body = bytearray(rng.choice(alphabet) for _ in range(size))
        p = rng.choice(pats)
        for at in (size - len(p), 29 - len(p) % 3, 61, 94, 127):  # packet end, group offsets 29..31
            if 0 <= at <= size - len(p):
                body[at:at + len(p)] = p
        q = rng.choice(pats)
        if i % 5 == 0 and size > 40:  # a NUL right after, right before and inside a start
            at = rng.randrange(8, size - len(q) - 8)
            body[at:at + len(q)] = q
            body[at + (i // 5) % 3 - 1 + (len(q) if i % 2 else 0)] = 0
        pkts.append(bytes(body))
    return pkts


@pytest.fixture(scope="module")
def finder(tmp_path_factory):
    return RefFinder(str(tmp_path_factory.mktemp("kmp_find_ref")))


@pytest.fixture(scope="module")
def engines():
    u, p = kmp.Matcher(0, engine="union"), kmp.Matcher(0, engine="perpat")
    yield u, p
    u.close()
    p.close()


def check_all(engines, oracle, finder, pats, pkts, label, gate):
    assert (gate_geometry(pats) is not None) == gate, label
    union, perpat = engines
    check_find(union, finder, pats, pkts, label=label)  # find forms vs the reference finder, counts vs records
    data, offsets = csr(pkts)
    want = oracle.count_csr(data, offsets, pats)
    assert union.count_host(data, offsets) == want, label
    perpat.set_patterns(pats)
    assert perpat.count_host(data, offsets) == want, label


def test_gate_geometry_of_strings(strings_txt):
    """strings.txt gets a gate of 1024 words (4 KB): it fits the block's shared memory next to the probe tables"""
    assert gate_geometry(kmp.load_patterns(strings_txt)) == (1024, 22)
    assert gate_geometry([b"a", b"abc"]) is None
    assert gate_geometry([bytes([a, b]) for a in range(1, 256) for b in range(1, 10)]) is None


@pytest.mark.gpu
def test_colliding_keys(engines, oracle, finder):
    rng = random.Random(0x6A7E)
    alphabet = bytes(range(0x20, 0x7F))
    pats = colliding_set(rng, alphabet)
    pkts = planted_packets(rng, pats, alphabet, 3000, 97)
    pkts += planted_packets(rng, pats, alphabet, 40, 2000)
    check_all(engines, oracle, finder, pats, pkts, "colliding", True)


@pytest.mark.gpu
def test_short_patterns_sharing_prefixes(engines, oracle, finder):
    rng = random.Random(23)
    alphabet = b"abcdeABCDE!#%\0"
    text = alphabet.replace(b"\0", b"")
    pats = [b"ab", b"abc", b"abcd", b"abcdeab", b"ba", b"bab", b"Ab", b"aB", b"abC", b"ABc", b"cd", b"cde", b"dc",
            b"dca", b"eA", b"eAe", b"!#", b"#%!", b"%%%%%%%%%", b"abcdeabcdeabcdeabcdeab"]
    # item ends: packets of 1400 bytes over more than a 64 KB work item, every one ending with a short pattern
    pkts = planted_packets(rng, pats, alphabet, 200, 1400)
    for i in range(2000):  # tiny packets: starts right after a packet boundary, 2- and 3-byte patterns filling them
        p = pats[i % len(pats)]
        pkts.append(p if i % 3 else p + bytes(rng.choice(text) for _ in range(i % 7)))
    check_all(engines, oracle, finder, pats, pkts, "prefixes", True)
    # one-byte patterns too: no gate
    check_all(engines, oracle, finder, pats + [b"a", b"E"], pkts, "prefixes+1", False)


@pytest.mark.gpu
def test_nul_and_packet_edges(engines, oracle, finder):
    pats = [b"id", b"ack", b"ttl", b"http", b"xid"]
    pkts = []
    for p in pats:
        for lead in range(0, 40):
            pkts.append(b"." * lead + p)                       # ends at the packet's end
            pkts.append(b"." * lead + p + b"\0" + p)           # right before a NUL; after it (cut)
            pkts.append(b"." * lead + p[:-1] + b"\0" + p[-1:])  # a NUL inside the start
            pkts.append(b"." * lead + b"\0" + p)               # right after a NUL (cut)
            pkts.append(b"." * lead + p[:1])                   # cut by the packet boundary, the rest in the next
            pkts.append(p[1:] + b"." * lead)
    check_all(engines, oracle, finder, pats, pkts, "nul", True)


@pytest.mark.gpu
def test_group_offsets_29_to_31(engines, oracle, finder):
    rng = random.Random(29)
    pats = [b"qz", b"qzx", b"zxq", b"xq", b"zqzqzqzqzqzq", b"zzx"]
    pkts = []
    for size in (64, 96, 128, 4096):
        for at in range(size):
            if at % 32 >= 29:
                body = bytearray(b"-" * size)
                p = pats[at % len(pats)]
                body[at:at + len(p)] = p[: size - at]
                pkts.append(bytes(body))
    pkts.append(bytes(rng.choice(b"qzx-") for _ in range(70000)))
    check_all(engines, oracle, finder, pats, pkts, "offsets", True)


@pytest.mark.gpu
def test_high_bytes(engines, oracle, finder):
    rng = random.Random(0x80)
    alphabet = bytes(range(0x61, 0x65)) + bytes(range(0x80, 0x88)) + bytes(range(0xE0, 0xE6)) + b"\xff"
    pats = [bytes([0x80, 0xFF]), bytes([0xE1, 0x61]), bytes([0x61, 0xE1, 0x81]), bytes([0x61, 0xE1, 0x61]),
            bytes([0xFF, 0xFF, 0xE1, 0x80]), bytes([0x81, 0x82, 0x83, 0x84, 0x85]), bytes([0xE3, 0x63, 0x83])]
    pkts = planted_packets(rng, pats, alphabet, 2000, 150)
    check_all(engines, oracle, finder, pats, pkts, "high", True)


@pytest.mark.gpu
def test_no_gate_for_large_sets(engines, oracle, finder):
    rng = random.Random(4096)
    alphabet = bytes(range(0x30, 0x5B))
    pats = sorted({bytes(rng.choice(alphabet) for _ in range(2)) for _ in range(900)})
    pats += [bytes(rng.choice(alphabet) for _ in range(rng.randint(3, 20))) for _ in range(200)]
    pkts = planted_packets(rng, pats, alphabet, 2000, 300)
    check_all(engines, oracle, finder, pats, pkts, "large", False)
