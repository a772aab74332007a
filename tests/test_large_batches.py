"""Batches past 4 GiB and packets at the size limit, against exact answers.

The union kernel keeps a candidate's absolute position in 56 bits (low word + high bits next to its room), looks a
packet up from the low words of `offsets` relative to the item's first row, picks 64, 128 or 256 KiB work items by the
batch's span, and the find path sorts on (position - first_byte) << pbits | pattern.  All of that only runs differently
once a batch crosses 2^32 (or 4 / 8 GiB of span), so these tests build one ~9.3 GiB stream on the device and check every
count and find form on spans of it, and a packet of the largest size the library accepts.

The stream.  Background bytes are 0x80..0xFF; no pattern holds any of them, so every match lies inside a planted window:
  - a two-byte marker ("id") at a seeded offset of every packet of two bytes or more;
  - islands of 64..2048 bytes of the patterns' alphabet, with NULs and planted patterns, at random places and at
    deliberate ones: around 2^32 and 2^33 (+-1, +-31), a 99-byte pattern (which holds the 40- and 17-byte ones)
    straddling 2^32 inside a packet that straddles it, a match ending exactly at that packet's end, a NUL at 2^33 - 1
    inside the 40 MB packet that straddles 2^33 (it kills the rest of that packet), and the first and last bytes of
    every span.
The expected records: each packet's windows are cut at its bounds and at its first NUL and run through the reference
finder as mini-packets, whose records are shifted back; a marker alone in its packet is the reference's records of
"id", shifted.  Nothing of the 9.3 GiB is scanned on the host, and a packet skipped or scanned twice shows up."""
import math
import struct
from types import SimpleNamespace

import numpy as np
import pytest

from kmpb_harness import DeviceBatch, udp_frame
from kmpb_reference import finder, firsts, keys

import multithreading_string_matching_b200 as kmp

pytestmark = pytest.mark.gpu

GiB, MiB = 1 << 30, 1 << 20
X1, X2 = 1 << 32, 1 << 33
N = 10_000_000_000        # bytes in the stream (9.31 GiB: the whole-stream span takes 256 KiB work items)
LIMIT = (1 << 31) - (1 << 20)  # a packet must be shorter (include/kmpb200.h, KMPB_PACKET_LIMIT)
MARK = b"id"
ELIMIT = -8
SEED = 20261020


# ---- pattern set ------------------------------------------------------------------------------------

def long_patterns():
    """99 bytes whose index 50 lands on 2^32 when planted at 2^32 - 50: "ack" at 2^32 - 31, "rrrr" at 2^32 - 1 .. 2^32 + 2,
    "http" at 2^32 + 31; the 40- and 17-byte patterns are slices of it that straddle 2^32 as well"""
    rng = np.random.default_rng(SEED + 99)
    p99 = bytearray(rng.choice(np.frombuffer(b"abcdefghjklmnopsuvwxyz0123456789_-", np.uint8), 99).tobytes())
    p99[19:22] = b"ack"
    p99[49:53] = b"rrrr"
    p99[81:85] = b"http"
    p99 = bytes(p99)
    return p99[42:59], p99[30:70], p99


def pattern_set(strings):
    p17, p40, p99 = long_patterns()
    pats = list(strings) + [b"d", p17, p40, p99]
    assert all(0 < b < 0x80 for p in pats for b in p)  # so no match can touch the background
    assert MARK in pats
    return pats


def key_counts(k, patterns):
    hist = np.bincount((k & np.uint64(1023)).astype(np.int64), minlength=len(patterns))
    return [int(hist[f]) for f in firsts(patterns)]


# ---- the planted content ----------------------------------------------------------------------------

class Plan:
    """What a buffer holds besides its background: markers (absolute positions of "id") and islands (absolute start,
    bytes), merged into standalone markers and non-touching windows whose final bytes are known."""

    def __init__(self, markers, islands):
        markers = np.asarray(markers, dtype=np.int64)
        st = np.concatenate([markers, np.array([s for s, _ in islands], dtype=np.int64)])
        en = np.concatenate([markers + len(MARK), np.array([s + len(b) for s, b in islands], dtype=np.int64)])
        who = np.concatenate([np.full(len(markers), -1, dtype=np.int64), np.arange(len(islands), dtype=np.int64)])
        order = np.argsort(st, kind="stable")
        st, en, who = st[order], en[order], who[order]
        reach = np.maximum.accumulate(en)
        new = np.ones(len(st), dtype=bool)
        new[1:] = st[1:] > reach[:-1]  # touching intervals merge: a match could run from one into the other
        heads = np.flatnonzero(new)
        tails = np.append(heads[1:], len(st))
        alone = (tails - heads == 1) & (who[heads] < 0)
        self.markers = st[heads[alone]]
        self.all_markers = markers
        self.windows = []  # (start, bytes), sorted, separated by background
        for h, t in zip(heads[~alone], tails[~alone]):
            w0 = int(st[h])
            buf = bytearray(int(reach[t - 1]) - w0)
            for j in range(h, t):  # markers first, then the islands in the order they were planted
                if who[j] < 0:
                    buf[st[j] - w0: st[j] - w0 + len(MARK)] = MARK
            for j in sorted(range(h, t), key=lambda j: who[j]):
                if who[j] >= 0:
                    s, b = islands[who[j]]
                    buf[s - w0: s - w0 + len(b)] = b
            self.windows.append((w0, bytes(buf)))

    def write(self, d_bytes, seed):
        """background, markers, windows -> the device buffer"""
        import torch

        block = torch.from_numpy(np.random.default_rng(seed).integers(0x80, 0x100, (1 << 20) + 7, dtype=np.uint8)).cuda()
        n, b = d_bytes.numel(), block.numel()
        reps = n // b
        d_bytes[: reps * b].view(reps, b).copy_(block.expand(reps, b))
        d_bytes[reps * b:] = block[: n - reps * b]
        at = torch.from_numpy(self.all_markers).cuda()
        for i, c in enumerate(MARK):
            d_bytes[at + i] = c
        del at
        if self.windows:
            starts = np.array([s for s, _ in self.windows], dtype=np.int64)
            lens = np.array([len(w) for _, w in self.windows], dtype=np.int64)
            idx = np.repeat(starts - np.concatenate([[0], np.cumsum(lens)[:-1]]), lens) + np.arange(lens.sum(), dtype=np.int64)
            vals = np.frombuffer(b"".join(w for _, w in self.windows), dtype=np.uint8)
            d_bytes[torch.from_numpy(idx).cuda()] = torch.from_numpy(vals.copy()).cuda()
        torch.cuda.synchronize()

    def expect(self, offsets, patterns):
        """sorted record keys of the batch `offsets` (absolute, packets numbered from 0) over this content"""
        offsets = np.asarray(offsets, dtype=np.uint64)
        off = offsets.astype(np.int64)
        n, lo, hi = len(off) - 1, int(off[0]), int(off[-1])
        # every window cut at packet bounds
        pieces, pk, po = [], [], []
        nul = {}
        for w0, w in self.windows:
            w1 = w0 + len(w)
            if w1 <= lo or w0 >= hi:
                continue
            k = max(int(np.searchsorted(off, max(w0, lo), "right")) - 1, 0)
            while k < n and off[k] < w1:
                ps, pe = int(off[k]), int(off[k + 1])
                a, b = max(w0, ps), min(w1, pe)
                if a < b:
                    piece = w[a - w0: b - w0]
                    z = piece.find(b"\0")
                    if z >= 0:
                        nul[k] = min(nul.get(k, 1 << 62), a + z)
                    pieces.append(piece)
                    pk.append(k)
                    po.append(a - ps)
                k += 1
        # the text of a packet ends at its first NUL: pieces that start after it hold nothing
        keep = [i for i in range(len(pieces)) if off[pk[i]] + po[i] < nul.get(pk[i], 1 << 62)]
        parts = []
        if keep:
            data = np.frombuffer(b"".join(pieces[i] for i in keep), dtype=np.uint8)
            cut = np.zeros(len(keep) + 1, dtype=np.uint64)
            np.cumsum([len(pieces[i]) for i in keep], out=cut[1:])
            r = finder().find_csr(data, cut, patterns)
            kk = np.array([pk[i] for i in keep], dtype=np.uint64)
            oo = np.array([po[i] for i in keep], dtype=np.uint64)
            j = r["packet"].astype(np.int64)
            parts.append(keys({"packet": kk[j], "offset": oo[j] + r["offset"], "pattern": r["pattern"]}))
        # markers alone in their packet: the records of "id", shifted, unless a NUL comes before them
        m = self.markers[(self.markers >= lo) & (self.markers < hi)]
        if m.size:
            k = np.searchsorted(off, m, "right") - 1
            assert (m + len(MARK) <= off[k + 1]).all(), "a standalone marker crosses a packet boundary"
            nul_at = np.full(n, 1 << 62, dtype=np.int64)
            for kn, z in nul.items():
                nul_at[kn] = z
            alive = nul_at[k] > m
            k, m = k[alive], m[alive]
            t = finder().find_csr(np.frombuffer(MARK, np.uint8), np.array([0, len(MARK)], np.uint64), patterns)
            for ro, rp in zip(t["offset"].tolist(), t["pattern"].tolist()):
                parts.append(keys({"packet": k, "offset": m - off[k] + ro, "pattern": np.full(k.size, rp)}))
        return np.sort(np.concatenate(parts)) if parts else np.zeros(0, dtype=np.uint64)


def island(rng, alpha, length, pool, nul):
    """`length` bytes of the alphabet with patterns of `pool` planted every few bytes, and one NUL if `nul`"""
    b = bytearray(alpha[rng.integers(0, len(alpha), length)].tobytes())
    at = int(rng.integers(0, 24))
    while at < length:
        p = pool[int(rng.integers(0, len(pool)))]
        if at + len(p) <= length:
            b[at:at + len(p)] = p
        at += len(p) + int(rng.integers(4, 60))
    if nul:
        b[int(rng.integers(0, length))] = 0
    return bytes(b)


def sizes_until(parts, pos, until, draw):
    """append packet sizes from draw(n) until the stream reaches `until`; returns the new end"""
    while pos < until:
        s = draw(8192).astype(np.int64)
        c = pos + np.cumsum(s)
        j = int(np.searchsorted(c, until))
        take = s[: j + 1] if j < len(s) else s
        parts.append(take)
        pos = int(c[len(take) - 1])
    return pos


def with_len_at_least(off, k, step, n=200):
    """first packet index from k on (step +1) or packet end from k down (step -1) whose packet has >= n bytes"""
    while off[k + 1] - off[k] < n if step > 0 else off[k] - off[k - 1] < n:
        k += step
    return k


# ---- fixtures -------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def patterns(strings_txt):
    return pattern_set(kmp.load_patterns(strings_txt))


@pytest.fixture(scope="module")
def matcher(patterns):
    m = kmp.Matcher(0, engine="union")
    m.set_patterns(patterns)
    yield m
    m.close()


def host_available():
    with open("/proc/meminfo") as f:
        for line in f:
            if line.startswith("MemAvailable:"):
                return int(line.split()[1]) * 1024
    return 0


def need_device(nbytes):
    import torch

    free, _ = torch.cuda.mem_get_info()
    if free < nbytes:
        pytest.skip("needs %.1f GiB of free device memory" % (nbytes / GiB))


def build_stream(patterns):
    """The ~9.3 GiB stream's layouts over the same bytes -- A (packets straddle 2^32 and 2^33), B (A cut at exactly 2^32
    and 2^33), C (A with the packet before the one straddling 2^32 merged into it, so that a NUL 1.1 MB below 2^32 ends
    that packet's text) -- the spans checked, the planted content and the expected records (host only)."""
    rng = np.random.default_rng(SEED)
    mixed = lambda n: np.where(rng.random(n) < 0.05, 0, rng.integers(1, 9001, n))  # noqa: E731
    parts, pos = [], 0
    n_eq = (3 * GiB // 2) // 1400
    parts.append(np.full(n_eq, 1400, dtype=np.int64))  # equal packets: the packet lookup is a division
    pos = sizes_until(parts, n_eq * 1400, n_eq * 1400 + 48 * MiB, lambda n: rng.integers(0, 65, n))  # items of many packets
    pos = sizes_until(parts, pos, X1 - 1_100_000, mixed)  # mixed sizes, empty packets: the search in `offsets`
    big_pk = [(pos, X1 + 7777)]  # ~1.1 MB straddling 2^32, ending just past it
    parts.append(np.array([X1 + 7777 - pos]))
    pos = X1 + 7777
    for until, size in ((X1 + 1200 * MiB, 7_000_003), (X1 + 2500 * MiB, 3_000_001)):
        pos = sizes_until(parts, pos, until, mixed)
        big_pk.append((pos, pos + size))
        parts.append(np.array([size]))
        pos += size
    pos = sizes_until(parts, pos, X2 - 13_000_000, mixed)
    big_pk.append((pos, X2 + 27_000_003))  # ~40 MB straddling 2^33
    parts.append(np.array([X2 + 27_000_003 - pos]))
    pos = sizes_until(parts, X2 + 27_000_003, N - 12_000, mixed)
    parts.append(np.array([N - pos]))
    sizes = np.concatenate(parts).astype(np.int64)
    off_a = np.zeros(len(sizes) + 1, dtype=np.uint64)
    np.cumsum(sizes, out=off_a[1:])
    assert off_a[-1] == N
    oa = off_a.astype(np.int64)
    cut = np.searchsorted(oa, [X1, X2])
    off_b = np.insert(off_a, cut, np.array([X1, X2], dtype=np.uint64))  # layout B: packet boundaries at 2^32, 2^33
    ob = off_b.astype(np.int64)
    kb1 = int(np.searchsorted(ob, X1))
    assert ob[kb1] == X1 and ob[kb1 + 1] > X1
    p1_start = big_pk[0][0]
    off_c = off_a[oa != p1_start]  # layout C: byte p1_start - 1 (a NUL) and the packet straddling 2^32 are one packet
    oc = off_c.astype(np.int64)
    kc0 = with_len_at_least(oc, int(np.searchsorted(oc, X1 - 32 * MiB)), 1)
    kc1 = with_len_at_least(oc, int(np.searchsorted(oc, X1 + 32 * MiB)), -1)

    # spans: (name, layout, k0, k1)
    n_a = len(oa) - 1
    k = int(np.searchsorted(oa, 7 * GiB // 2))
    while oa[k] % 2 == 0 or oa[k + 1] - oa[k] < 200:
        k += 1
    k1 = with_len_at_least(oa, int(np.searchsorted(oa, oa[k] + 5 * GiB)), -1)
    k_hi = with_len_at_least(oa, int(np.searchsorted(oa, X2 + 64 * MiB)), 1)
    k_hi1 = with_len_at_least(oa, int(np.searchsorted(oa, oa[k_hi] + GiB)), -1)
    k_3g = with_len_at_least(oa, int(np.searchsorted(oa, 3 * GiB)), -1)
    spans = {
        "whole": ("a", 0, n_a),
        "5GiB_odd_start": ("a", k, k1),
        "from_2^32": ("b", kb1, len(ob) - 1),
        "1GiB_above_2^33": ("a", k_hi, k_hi1),
        "first_3GiB": ("a", 0, k_3g),
        "nul_below_2^32": ("c", kc0, kc1),
    }
    layouts = {"a": oa, "b": ob, "c": oc}
    for name, (lay, s0, s1) in spans.items():
        o = layouts[lay]
        assert s0 < s1 and o[s1] - o[s1 - 1] >= 200 and o[s0 + 1] - o[s0] >= 200, name
    assert oa[k] < X1 and oa[k1] > X2 and 4 * GiB <= oa[k1] - oa[k] < 8 * GiB
    assert oa[k_hi] >> 32 == 2 and oa[k_hi1] >> 32 == 2
    assert ob[-1] - ob[kb1] >= 4 * GiB

    # markers: one per packet of two bytes or more (layout A)
    la = np.diff(oa)
    with2 = np.flatnonzero(la >= 2)
    markers = oa[with2] + (rng.random(len(with2)) * (la[with2] - 1)).astype(np.int64)

    alpha = np.array(sorted(set(b"".join(patterns))), dtype=np.uint8)
    pool = [p for p in patterns if p != b"d"] + list(long_patterns()) * 8
    p17, p40, p99 = long_patterns()
    # no NUL where it would kill a deliberate plant: the packet straddling 2^32, the 40 MB packet before 2^33 - 1, and
    # the first and last packets of every span
    guard = [big_pk[0], (big_pk[-1][0], X2)]
    for lay, s0, s1 in spans.values():
        o = layouts[lay]
        guard += [(int(o[s0]), int(o[s0 + 1])), (int(o[s1 - 1]), int(o[s1]))]
    guard = np.array(guard, dtype=np.int64)

    def guarded(a, b):
        return bool(((guard[:, 0] < b) & (a < guard[:, 1])).any())

    islands = []
    starts = list(rng.integers(0, N - 4096, 24_000))
    for s, e in big_pk:  # interiors of the big packets: no markers there, so an island every 128 KiB
        starts += list(range(s + 4321, e - 4096, 128 << 10))
    for s in starts:
        s = int(s)
        length = int(math.exp(rng.uniform(math.log(64), math.log(2048))))
        islands.append((s, island(rng, alpha, length, pool, rng.random() < 0.4 and not guarded(s, s + length))))
    # deliberate places (planted last: they win where a random island overlaps them)
    filler = lambda n: bytes(alpha[rng.integers(0, len(alpha), n)])  # noqa: E731
    islands.append((X1 - 60, filler(10) + p99 + filler(11)))  # p99[50] at 2^32
    e1 = big_pk[0][1]
    islands.append((e1 - 40, filler(40 - 17) + p17 + filler(40)))  # a long match ending exactly at the packet's end
    x2 = bytearray(filler(80))  # [2^33 - 40, 2^33 + 40): NUL at 2^33 - 1
    x2[9:12] = b"ack"
    x2[39] = 0
    x2[40:43] = b"rrr"
    x2[71:75] = b"http"
    islands.append((X2 - 40, bytes(x2)))
    islands.append((p1_start - 1, b"\0http" + filler(20)))  # NUL just before the packet straddling 2^32 (C: inside it)
    for lay, s0, s1 in spans.values():
        o = layouts[lay]
        fb, eb = int(o[s0]), int(o[s1])
        if fb != X1:
            islands.append((fb, p17 + filler(47)))
        islands.append((eb - 64, filler(24) + p40))
    plan = Plan(markers, islands)

    g = SimpleNamespace(plan=plan, layouts=layouts, spans=spans, big_packets=big_pk)
    whole = plan.expect(off_a, patterns)
    g.want = {}
    for name, (lay, s0, s1) in spans.items():
        if lay == "a":
            pk = whole >> np.uint64(41)
            sel = whole[(pk >= s0) & (pk < s1)]
            g.want[name] = sel - (np.uint64(s0) << np.uint64(41))
        else:
            g.want[name] = plan.expect(layouts[lay][s0:s1 + 1].astype(np.uint64), patterns)
    return g


@pytest.fixture(scope="module")
def big(patterns):
    import torch

    need_device(13 * GiB)
    g = build_stream(patterns)
    g.d_bytes = torch.empty(N + 4096, dtype=torch.uint8, device="cuda:0")
    g.plan.write(g.d_bytes, SEED)
    g.batch = {lay: DeviceBatch.on_device(g.d_bytes, torch.from_numpy(o).cuda(), o) for lay, o in g.layouts.items()}
    yield g
    del g.d_bytes, g.batch
    torch.cuda.empty_cache()


def diff(got, want):
    g, w = set(got.tolist()), set(want.tolist())
    dec = lambda ks: [(k >> 41, (k >> 10) & (2**31 - 1), k & 1023) for k in sorted(ks)[:5]]  # noqa: E731
    return "%d got, %d expected; missing %s; extra %s" % (len(got), len(want), dec(w - g), dec(g - w))


def check_all_forms(m, patterns, batch, k0, k1, want, label, perpat=True):
    """count (union, per-pattern), find unsorted, sorted, and sorted into a buffer one record short"""
    counts = key_counts(want, patterns)
    assert len(want) > 0
    assert batch.count(m, k0=k0, k1=k1) == [counts], (label, "union counts")
    if perpat:
        m.set_engine("perpat")
        try:
            assert batch.count(m, k0=k0, k1=k1) == [counts], (label, "perpat counts")
        finally:
            m.set_engine("union")
    total = len(want)
    rec, n, ok = batch.find(m, total, False, k0, k1, canary=64)
    got = np.sort(keys(rec))
    assert n == total and ok and np.array_equal(got, want), (label, "unsorted", diff(got, want))
    rec, n, ok = batch.find(m, total, True, k0, k1, canary=64)
    got = keys(rec)
    assert n == total and ok and np.array_equal(got, want), (label, "sorted", diff(got, want))
    rec, n, ok = batch.find(m, total - 1, True, k0, k1, canary=64)
    got = np.sort(keys(rec))
    at = np.minimum(np.searchsorted(want, got), total - 1)
    assert n == total and ok and len(got) == total - 1, (label, "capacity - 1", n)
    assert (np.diff(got) > 0).all() and (want[at] == got).all(), (label, "capacity - 1: not a distinct subset")
    kmp.matcher.check(kmp.lib().kmpb_check_device_errors(m.handle))


# ---- packets at the size limit (own 2 GiB buffer: runs before the big stream is built) ----------------

@pytest.fixture(scope="class")
def limit_batch(patterns):
    """~2 GiB buffer around a packet of LIMIT - 1 bytes, its host copy, and a context of its own: the host forms grow
    the context's four staging slots to the size of that packet, and closing it gives their 8 GiB back"""
    import torch

    nbytes = 300 * 1024 + LIMIT + 64 * 1024
    need_device(13 * GiB)
    if host_available() < nbytes + 4 * GiB:
        pytest.skip("needs %.1f GiB of host memory" % ((nbytes + 4 * GiB) / GiB))
    rng = np.random.default_rng(SEED + 4)
    parts = []
    s_g = sizes_until(parts, 0, 150 * 1024, lambda n: np.where(rng.random(n) < 0.1, 0, rng.integers(1, 9001, n)))
    e_g = s_g + LIMIT - 1
    tail = [5000, 0, 1, 9000, 777, 3000]
    sizes = np.concatenate(parts + [np.array([LIMIT - 1] + tail)]).astype(np.int64)
    off = np.zeros(len(sizes) + 1, dtype=np.uint64)
    np.cumsum(sizes, out=off[1:])
    g_index = len(sizes) - len(tail) - 1
    assert off[g_index] == s_g and off[g_index + 1] == e_g and off[-1] + 4096 <= nbytes
    o = off.astype(np.int64)
    la = np.diff(o)
    with2 = np.flatnonzero(la >= 2)
    markers = o[with2] + (rng.random(len(with2)) * (la[with2] - 1)).astype(np.int64)
    alpha = np.array(sorted(set(b"".join(patterns))), dtype=np.uint8)
    p17, p40, p99 = long_patterns()
    pool = [p for p in patterns if p != b"d"]
    islands = [(int(s), island(rng, alpha, 400, pool, True)) for s in rng.integers(0, s_g - 400, 40)]
    islands += [(int(s), island(rng, alpha, 400, pool, True)) for s in rng.integers(e_g, int(o[-1]) - 400, 6)]
    islands.append((s_g, p17 + island(rng, alpha, 200, pool, False)))          # the packet's first byte
    islands.append((s_g + (1 << 24) + 12345, island(rng, alpha, 900, pool + [p99], False)))  # past 2^24: the float division
    islands.append((s_g + GiB + 777, island(rng, alpha, 2000, pool + [p40], False)))
    islands.append((e_g - 300, island(rng, alpha, 300 - 40, pool, False) + p40))  # ending exactly at its end
    lb = SimpleNamespace(plan=Plan(markers, islands), off=off, g=g_index)
    lb.d_bytes = torch.empty(nbytes, dtype=torch.uint8, device="cuda:0")
    lb.plan.write(lb.d_bytes, SEED + 4)
    lb.host = lb.d_bytes.cpu().numpy()
    lb.m = kmp.Matcher(0, engine="union")
    lb.m.set_patterns(patterns)
    yield lb
    lb.m.close()
    lb.d_bytes = lb.host = lb.m = None
    torch.cuda.empty_cache()


class TestPacketLimit:
    """A packet of LIMIT - 1 bytes works in every form; one of LIMIT bytes is refused (one 2 GiB buffer for both)."""

    def test_packet_one_byte_under_the_limit(self, patterns, limit_batch):
        """A packet of LIMIT - 1 bytes behind ~150 KiB of small packets and before a few more, and the same packet alone:
        exact counts and records through the device forms, kmpb_count_host and kmpb_find_host, and no KMPB_ELIMIT."""
        import torch

        lb = limit_batch
        matcher, plan, d_bytes, host, off, g = lb.m, lb.plan, lb.d_bytes, lb.host, lb.off, lb.g
        cases = {"with neighbours": off, "alone": off[g:g + 2]}
        for label, offs in cases.items():
            want = plan.expect(offs, patterns)
            counts = key_counts(want, patterns)
            assert len(want) > 100 and counts[patterns.index(long_patterns()[1])] >= 1, label
            batch = DeviceBatch.on_device(d_bytes, torch.from_numpy(offs.astype(np.int64)).cuda(), offs)
            check_all_forms(matcher, patterns, batch, 0, len(offs) - 1, want, label, perpat=False)
            assert matcher.count_host(host, offs) == counts, label
            got = keys(matcher.find_host(host, offs))
            assert np.array_equal(got, want), (label, "find_host", diff(got, want))

    def test_packet_at_the_limit_is_refused(self, limit_batch):
        """A packet of LIMIT bytes: KMPB_ELIMIT from the host forms (before anything runs) and from
        kmpb_check_device_errors after a device form; the check reports it once."""
        import torch

        lb = limit_batch
        matcher, d_bytes, host, off, g = lb.m, lb.d_bytes, lb.host, lb.off, lb.g
        s = int(off[g])
        for offs in (np.array([s, s + LIMIT], dtype=np.uint64), np.concatenate([off[:g + 1], [s + LIMIT]]).astype(np.uint64)):
            for call in (matcher.count_host, matcher.find_host):
                with pytest.raises(kmp.KmpbError) as e:
                    call(host, offs)
                assert e.value.code == ELIMIT and "packet %d " % (len(offs) - 2) in str(e.value), str(e.value)
            DeviceBatch.on_device(d_bytes, torch.from_numpy(offs.astype(np.int64)).cuda(), offs).count(matcher)
            lib = kmp.lib()
            assert lib.kmpb_check_device_errors(matcher.handle) == ELIMIT
            assert lib.kmpb_check_device_errors(matcher.handle) == 0
        # a batch within the limits afterwards: clean
        DeviceBatch.on_device(d_bytes, torch.from_numpy(off.astype(np.int64)).cuda(), off).count(matcher)
        kmp.matcher.check(kmp.lib().kmpb_check_device_errors(matcher.handle))


# ---- the ~9.3 GiB stream --------------------------------------------------------------------------

@pytest.mark.parametrize("name", ["whole", "5GiB_odd_start", "from_2^32", "1GiB_above_2^33", "first_3GiB", "nul_below_2^32"])
def test_device_spans(matcher, patterns, big, name):
    """Every device form on a span of the stream (a shifted d_offsets + span=), packets numbered from the span's
    first: whole (256 KiB items), 5 GiB from an odd first byte near 3.5 GiB across 2^32 and 2^33 (128 KiB items), a
    slice that starts exactly at 2^32, 1 GiB above 2^33 (high word 2 everywhere), the first 3 GiB (64 KiB items)."""
    lay, k0, k1 = big.spans[name]
    check_all_forms(matcher, patterns, big.batch[lay], k0, k1, big.want[name], name)


def test_plants_are_where_they_should_be(patterns, big):
    """The deliberate plants are among the expected records (so the spans above do test them) -- and the ones a NUL
    kills are not."""
    p17, p40, p99 = long_patterns()
    ib = big.spans["from_2^32"][1:]
    oa, ob = big.layouts["a"], big.layouts["b"]

    def at(layout, want, pos, pat, k_base=0):
        o = big.layouts[layout]
        k = int(np.searchsorted(o, pos, "right")) - 1
        key = keys({"packet": [k - k_base], "offset": [pos - int(o[k])], "pattern": [patterns.index(pat)]})[0]
        i = int(np.searchsorted(want, key))
        return i < len(want) and want[i] == key

    wa, wb, wc = big.want["whole"], big.want["from_2^32"], big.want["nul_below_2^32"]
    kb, kc = ib[0], big.spans["nul_below_2^32"][1]
    s1 = big.big_packets[0][0]
    assert at("a", wa, s1, b"http")
    for pos, pat in ((s1, b"http"), (X1 - 50, p99), (X1 - 1, b"rr"), (X1, b"rr"), (X1 + 31, b"http"),
                     (big.big_packets[0][1] - 17, p17)):
        assert not at("c", wc, pos, pat, kc), (hex(pos), pat)  # after the NUL at s1 - 1, 1.1 MB below 2^32
    for pos, pat in ((X1 - 50, p99), (X1 - 20, p40), (X1 - 8, p17), (X1 - 31, b"ack"), (X1 - 1, b"rr"), (X1, b"rr"),
                     (X1 + 1, b"rr"), (X1 + 31, b"http"), (big.big_packets[0][1] - 17, p17), (X2 - 31, b"ack")):
        assert at("a", wa, pos, pat), (hex(pos), pat)
    for pos, pat in ((X2, b"rr"), (X2 + 1, b"rr"), (X2 + 31, b"http")):
        assert not at("a", wa, pos, pat), (hex(pos), pat)  # after the NUL at 2^33 - 1 in the packet straddling 2^33
        assert at("b", wb, pos, pat, kb), (hex(pos), pat)  # ... which layout B cuts at 2^33
    for pos, pat in ((X1, b"rr"), (X1 + 1, b"rr"), (X1 + 31, b"http")):
        assert at("b", wb, pos, pat, kb)
    assert len(oa) + 2 == len(ob)


def test_host_forms_past_4GiB(matcher, patterns, big):
    """kmpb_count_host and kmpb_find_host on a pageable host copy of the 5 GiB span across 2^32 and 2^33, offsets
    absolute from 0: its chunks start above 2^32."""
    lay, k0, k1 = big.spans["5GiB_odd_start"]
    o = big.layouts[lay]
    base = int(o[k0]) & ~511
    if host_available() < (int(o[k1]) - base) + 4 * GiB:
        pytest.skip("needs %.1f GiB of host memory" % ((int(o[k1]) - base + 4 * GiB) / GiB))
    host = big.d_bytes[base:int(o[k1])].cpu().numpy()
    offs = np.ascontiguousarray(o[k0:k1 + 1].astype(np.uint64))
    want = big.want["5GiB_odd_start"]
    # absolute byte 0, below the copy: the library reads a chunk from bytes + (offsets[k0] & ~511) on, never below
    ptr = host.ctypes.data - base
    assert matcher.count_host_ptr(ptr, offs.ctypes.data, k1 - k0) == key_counts(want, patterns)
    got = keys(matcher.find_host_ptr(ptr, offs.ctypes.data, k1 - k0, len(want) + 16))
    assert np.array_equal(got, want), diff(got, want)
    del host


def test_tables_in_global_memory(patterns, big):
    """~700 patterns (the probe tables leave shared memory), most of them cut from the planted windows, on the span
    above 2^33: counts and sorted records."""
    lay, k0, k1 = big.spans["1GiB_above_2^33"]
    o = big.layouts[lay]
    rng = np.random.default_rng(SEED + 700)
    wins = [w for w0, w in big.plan.windows if o[k0] <= w0 and w0 + len(w) <= o[k1] and len(w) >= 64]
    pats = list(patterns)
    while len(pats) < 700:
        w = wins[int(rng.integers(0, len(wins)))]
        m = int(rng.choice([2, 3, 4, 5, 8, 9, 17, 40]))
        at = int(rng.integers(0, len(w) - m + 1))
        if b"\0" not in w[at:at + m]:
            pats.append(w[at:at + m])
    pats += pats[100:110]  # duplicates: credited to their first listing
    want = big.plan.expect(o[k0:k1 + 1].astype(np.uint64), pats)
    with kmp.Matcher(0, engine="union") as m:
        m.set_patterns(pats)
        counts = key_counts(want, pats)
        assert big.batch[lay].count(m, k0=k0, k1=k1) == [counts]
        rec, n, ok = big.batch[lay].find(m, len(want), True, k0, k1, canary=64)
        got = keys(rec)
        assert n == len(want) and ok and np.array_equal(got, want), diff(got, want)


def test_savefile_and_stream_refuse_a_packet_at_the_limit(matcher, patterns, tmp_path):
    """The savefile forms and pushed frames check every payload before anything runs: one of LIMIT bytes (its frame's
    captured length less the headers) is refused by kmpb_count_pcap, kmpb_find_pcap and kmpb_stream_push, and the
    packets around it still count when the range leaves it out."""
    small = [udp_frame(b"xx http yy ack".ljust(100, b"\0")), udp_frame(b"dos udp test".ljust(50, b"\0"))]
    path = str(tmp_path / "giant.pcap")
    with open(path, "wb") as f:  # the giant payload is a hole in a sparse file: zeros
        f.write(struct.pack("<IHHiIII", 0xA1B2C3D4, 2, 4, 0, 0, 262144, 1))
        f.write(struct.pack("<IIII", 1, 2, len(small[0]), len(small[0])) + small[0])
        head = udp_frame(b"")
        f.write(struct.pack("<IIII", 1, 2, len(head) + LIMIT, len(head) + LIMIT) + head)
        f.seek(LIMIT, 1)
        f.write(struct.pack("<IIII", 1, 2, len(small[1]), len(small[1])) + small[1])
    for call in (lambda: matcher.count_pcap_streamed(path), lambda: matcher.find_pcap(path),
                 lambda: matcher.count_pcap_streamed(path, first=1, count=1)):
        with pytest.raises(kmp.KmpbError) as e:
            call()
        assert e.value.code == ELIMIT and "packet 1 " in str(e.value), str(e.value)
    data, offs = np.frombuffer(b"".join(fr[42:] for fr in small), np.uint8), np.array([0, 100, 150], np.uint64)
    want = matcher.count_host(data, offs)
    assert sum(want) > 0
    first = matcher.count_host(data, offs[:2])
    assert matcher.count_pcap_streamed(path, first=0, count=1) == first
    assert matcher.count_pcap_streamed(path, first=2, count=1) == [w - f for w, f in zip(want, first)]
    with matcher.stream("udp") as st:
        st.push(small[0])
        giant = udp_frame(bytes(LIMIT))
        with pytest.raises(kmp.KmpbError) as e:
            st.push(giant)
        assert e.value.code == ELIMIT and "packet 1 " in str(e.value), str(e.value)
        del giant
        st.push(small[1])
        assert st.flush() == want
    kmp.matcher.check(kmp.lib().kmpb_check_device_errors(matcher.handle))
