"""What the right answer is: the matching rules written down once, for every test module.  CPU only (no torch, no
device).

A pattern matches at every start of its bytes in a packet's text, which is the payload up to its first NUL; matches
overlap and never cross a packet's end.  A nocase pattern's matches are the case-sensitive matches of the folded
pattern in the folded text (ASCII A-Z to a-z; folding never creates or moves a NUL).  A windowed pattern (lo, hi)
matches only at offsets lo..hi.  Patterns that are equal in (folded bytes, flag, window) are one pattern: every listing
gets the full count, and a record carries the lowest index of them (`firsts`).

`naive` is the definition as code; `expected` derives the same answers from the reference finder
(tests/c/kmp_find_ref.c, a restatement of the reference's kmp_matcher that records where it hits) and `reference`
from numpy at the cost of a few table lookups per text byte.  The CPU tests cross-check the three."""
import ctypes
import functools
import os
import subprocess
import tempfile

import numpy as np

import multithreading_string_matching_b200 as kmp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORDER = ["packet", "offset", "pattern"]
FOLD_TABLE = np.array([c + 32 if 0x41 <= c <= 0x5A else c for c in range(256)], dtype=np.uint8)
LETTERS = set(range(0x41, 0x5B)) | set(range(0x61, 0x7B))


def csr(packets):
    offsets = np.zeros(len(packets) + 1, dtype=np.uint64)
    if packets:
        np.cumsum([len(p) for p in packets], out=offsets[1:])
    return np.frombuffer(b"".join(packets) + b"\0" * 16, dtype=np.uint8)[: int(offsets[-1])], offsets


def fold(b):
    return bytes(b).translate(FOLD_TABLE.tobytes())


def as_tuples(rec):
    return list(zip(rec["packet"].tolist(), rec["offset"].tolist(), rec["pattern"].tolist()))


def normalise(patterns, nocase=False, window=None):
    """(bytes, one flag each, one window or None each) from the shapes Matcher.set_patterns accepts"""
    patterns = [bytes(p) for p in patterns]
    n = len(patterns)
    nocase = [bool(x) for x in nocase] if isinstance(nocase, (list, tuple)) else [bool(nocase)] * n
    if window is None or (len(window) == 2 and all(isinstance(x, (int, np.integer)) for x in window)):
        window = [None if window is None else tuple(window)] * n
    else:
        window = [None if w is None else tuple(w) for w in window]
    return patterns, nocase, window


def firsts(patterns, nocase=False, window=None):
    """file-order index -> lowest index of an equal (folded bytes, flag, window)"""
    seen = {}
    return [seen.setdefault((fold(p) if n else p, n, w), i) for i, (p, n, w) in enumerate(zip(*normalise(patterns, nocase, window)))]


def naive(packets, patterns, nocase=False, window=None):
    """sorted (packet, offset, pattern) straight from the definition"""
    patterns, nocase, window = normalise(patterns, nocase, window)
    first = firsts(patterns, nocase, window)
    out = []
    for k, payload in enumerate(packets):
        text = payload.split(b"\0", 1)[0]
        for i, (p, n, w) in enumerate(zip(patterns, nocase, window)):
            if first[i] != i:
                continue
            t, q = (fold(text), fold(p)) if n else (text, p)
            out += [(k, s, i) for s in range(len(t) - len(q) + 1) if t[s:s + len(q)] == q and (w is None or w[0] <= s <= w[1])]
    return sorted(out)


class RefFinder:
    """ctypes view of tests/c/kmp_find_ref.c"""

    def __init__(self):
        cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"
        with tempfile.TemporaryDirectory(prefix="kmp_find_ref") as d:  # a loaded library outlives its file
            so = os.path.join(d, "libkmp_find_ref.so")
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


@functools.lru_cache(maxsize=None)
def finder():
    """the run's RefFinder: the C file is compiled once"""
    return RefFinder()


def expected(patterns, data, offsets, nocase=False, window=None, oracle=None):
    """(counts, sorted records, verdicts) from the reference finder: the records of each distinct pattern without its
    window (a nocase one: the folded pattern's in the folded text), those whose offset lies in its window, keyed to
    its first index; the counts are their histogram, the verdicts the packets they fall in.  With `oracle`, and no
    window in the set, the oracle's counts of each flag group must equal those counts."""
    patterns, nocase, window = normalise(patterns, nocase, window)
    n = len(patterns)
    first = firsts(patterns, nocase, window)
    data = np.ascontiguousarray(data, dtype=np.uint8)
    texts = {False: data}
    parts, ordered = [], True
    for nc in (False, True):
        own = [i for i in range(n) if nocase[i] == nc and first[i] == i]
        if not own:
            continue
        text = texts[nc] = FOLD_TABLE[data] if nc else data
        ks = [fold(patterns[i]) if nc else patterns[i] for i in own]
        r = finder().find_csr(text, offsets, ks)  # keyed to the first position in ks of an equal key
        if all(window[i] is None for i in own):  # distinct keys in file order: renumbering keeps the records sorted
            r["pattern"] = np.array(own, dtype=np.uint32)[r["pattern"].astype(np.int64)]
            parts.append(r)
            continue
        ordered = False  # (equal bytes under several windows: each owner takes the key's records in its window)
        r = r[np.argsort(r["pattern"], kind="stable")]
        bounds = np.searchsorted(r["pattern"], np.arange(len(ks) + 1))
        at = {}
        for j, (i, k) in enumerate(zip(own, ks)):
            f = at.setdefault(k, j)
            part = r[bounds[f]:bounds[f + 1]].copy()
            if window[i] is not None:
                part = part[(part["offset"] >= window[i][0]) & (part["offset"] <= window[i][1])]
            part["pattern"] = i
            parts.append(part)
    rec = np.concatenate(parts) if parts else np.zeros(0, dtype=kmp.MATCH_DTYPE)
    if len(parts) > 1 or not ordered:
        rec = rec[np.lexsort((rec["pattern"], rec["offset"], rec["packet"]))]
    hist = np.bincount(rec["pattern"].astype(np.int64), minlength=max(n, 1))
    counts = [int(hist[first[i]]) for i in range(n)]
    verdicts = np.zeros(len(offsets) - 1, dtype=bool)
    verdicts[rec["packet"].astype(np.int64)] = True
    if oracle is not None and all(w is None for w in window):
        for nc in (False, True):
            idx = [i for i in range(n) if nocase[i] == nc]
            if idx:
                got = oracle.count_csr(texts[nc], offsets, [fold(patterns[i]) if nc else patterns[i] for i in idx])
                assert got == [counts[i] for i in idx], ("the oracle's counts", nc)
    return counts, rec, verdicts


def assert_invariant(counts, rec, patterns):
    """for every pattern i, counts[i] = the records carrying i's first index"""
    first = firsts(patterns)
    hist = np.bincount(rec["pattern"].astype(np.int64), minlength=max(len(patterns), 1))
    assert [int(hist[first[i]]) for i in range(len(patterns))] == list(counts)


def keys(rec):
    """one sortable uint64 per record (or per entry of a mapping of the three fields' arrays): (packet, offset,
    pattern) order is key order"""
    packet, offset, pattern = (np.asarray(rec[f], dtype=np.uint64) for f in ORDER)
    if packet.size:
        assert int(packet.max()) < 1 << 23 and int(offset.max()) < 1 << 31 and int(pattern.max()) < 1 << 10
    return (packet << np.uint64(41)) | (offset << np.uint64(10)) | pattern


# ---- the numpy reference ---------------------------------------------------------------------------------------------

def _prefix64(text):
    """the little-endian 64-bit word of text bytes p..p+7 for every p (zero past the end)"""
    t = np.zeros(len(text) + 8, dtype=np.uint64)
    t[: len(text)] = text
    out = np.zeros(len(text), dtype=np.uint64)
    for i in range(8):
        out |= t[i: i + len(text)] << np.uint64(8 * i)
    return out


def reference(patterns, nocase, window, data, offsets):
    """(counts in file order, records sorted by (packet, offset, pattern), verdicts) of a set with windows.

    About one table lookup per (text position, distinct (flag, length)), not patterns x bytes: the distinct patterns
    are grouped by (flag, length); a group's keys are looked up at every text position with room for them (for a group
    of windowed patterns only at offsets [min lo, max hi]); the hits of a key, sorted by offset, give each of its
    patterns its records as one slice, cut by two binary searches on lo and hi."""
    patterns, nocase, window = normalise(patterns, nocase, window)
    data = np.ascontiguousarray(data, dtype=np.uint8)
    offsets = np.asarray(offsets, dtype=np.int64)
    starts, n_pk = offsets[:-1], len(offsets) - 1
    # a packet's text: its payload up to the first NUL
    nul = np.append(np.flatnonzero(data == 0), len(data))
    text_end = np.minimum(nul[np.searchsorted(nul, starts)], offsets[1:]) if n_pk else starts
    texts, words = {False: data, True: FOLD_TABLE[data]}, {}
    first = firsts(patterns, nocase, window)
    groups = {}
    for i, (p, nc, w) in enumerate(zip(patterns, nocase, window)):
        if first[i] == i:
            groups.setdefault((nc, len(p)), []).append((fold(p) if nc else p, w, i))
    rec_pk, rec_off, rec_pat = [], [], []
    for (nc, m), members in groups.items():
        windowed = all(w is not None for _, w, _ in members)
        o_lo = min(w[0] for _, w, _ in members) if windowed else 0
        o_hi = max(w[1] for _, w, _ in members) if windowed else 1 << 62
        first_pos = starts + o_lo
        cnt = np.maximum(np.minimum(text_end - m, starts + o_hi) - first_pos + 1, 0)
        total = int(cnt.sum())
        if total == 0:
            continue
        pk = np.repeat(np.arange(n_pk), cnt)
        pos = np.arange(total, dtype=np.int64) + np.repeat(first_pos - (np.cumsum(cnt) - cnt), cnt)
        text = texts[nc]
        if nc not in words:
            words[nc] = _prefix64(text)
        # the first min(m, 8) bytes as one word pick the candidates; longer keys are compared in full after that
        mask = np.uint64((1 << (8 * min(m, 8))) - 1)
        ks = sorted({k for k, _, _ in members})
        kw = np.array([int.from_bytes(k[:8], "little") for k in ks], dtype=np.uint64)
        kord = np.argsort(kw, kind="stable")
        sw = kw[kord]
        tw = words[nc][pos] & mask
        j = np.minimum(np.searchsorted(sw, tw), len(sw) - 1)
        cand = sw[j] == tw
        pk, pos = pk[cand], pos[cand]
        if m <= 8:
            kid = kord[j[cand]]  # (a key of up to 8 bytes is its word)
        else:
            skeys = np.array(ks, dtype="S%d" % m)
            tk = np.ascontiguousarray(np.lib.stride_tricks.sliding_window_view(text, m)[pos]).view("S%d" % m).ravel()
            kid = np.minimum(np.searchsorted(skeys, tk), len(ks) - 1)
            same = skeys[kid] == tk
            kid, pk, pos = kid[same], pk[same], pos[same]
        off = pos - starts[pk]
        order = np.lexsort((off, kid))
        kid, pk, off = kid[order], pk[order], off[order]
        bounds = np.searchsorted(kid, np.arange(len(ks) + 1))
        where = {k: x for x, k in enumerate(ks)}
        a_s, b_s, ids = [], [], []
        for key, w, i in members:
            a, b = bounds[where[key]], bounds[where[key] + 1]
            if w is not None:
                a, b = a + np.searchsorted(off[a:b], [w[0], w[1] + 1])
            a_s.append(a)
            b_s.append(b)
            ids.append(i)
        lens = np.array(b_s, dtype=np.int64) - np.array(a_s, dtype=np.int64)
        n = int(lens.sum())
        if n == 0:
            continue
        idx = np.arange(n, dtype=np.int64) + np.repeat(np.array(a_s, dtype=np.int64) - (np.cumsum(lens) - lens), lens)
        rec_pk.append(pk[idx])
        rec_off.append(off[idx])
        rec_pat.append(np.repeat(np.array(ids, dtype=np.int64), lens))
    rec = np.zeros(sum(len(x) for x in rec_pk), dtype=kmp.MATCH_DTYPE)
    if len(rec):
        pk, off, pat = (np.concatenate(x) for x in (rec_pk, rec_off, rec_pat))
        order = np.lexsort((pat, off, pk))
        rec["packet"], rec["offset"], rec["pattern"] = pk[order], off[order], pat[order]
    hist = np.bincount(rec["pattern"].astype(np.int64), minlength=max(len(patterns), 1))
    counts = [int(hist[first[i]]) for i in range(len(patterns))]
    verdicts = np.zeros(n_pk, dtype=bool)
    verdicts[rec["packet"].astype(np.int64)] = True
    return counts, rec, verdicts


# ---- the union kernel's prefix gate (automaton.c build_gate) ---------------------------------------------------------

GATE_MUL = 0x79B10000


def gate_slot(key, shift):
    return ((key * GATE_MUL) & 0xFFFFFFFF) >> shift


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
