#!/usr/bin/env python3
"""CPU model of the union engine's prefilter: candidate and event rates of different filter geometries on
the BASELINE workloads (no GPU).  A geometry = (depth, pattern buckets); a bucket's stage d passes the byte
values some member has at depth d (every value when a member is shorter).  Usage: scripts/filter_model.py
scripts/filter_model.py gate: the resolve step's prefix gate (automaton.c build_gate) on the C3 text -- candidates and
verification rounds per resolve step with the filter re-run, with the gate in its place, and with both (compare with
scripts/event_counts.py, which counts the same on a B200)."""
import sys, os, itertools, random
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from multithreading_string_matching_b200 import matcher as M

ALPHA = 96.0


def bucket_cost(members, depth):
    c = 1.0
    for d in range(depth):
        if any(len(p) <= d for p in members):
            continue
        c *= min(1.0, len({p[d] for p in members}) / ALPHA)
    return c if members else 0.0


def optimise(pats, depth, nb, seed=1):
    """contiguous DP split of the sorted patterns, then hill climbing (moves + swaps), as automaton.c does"""
    pats = sorted(set(pats), key=lambda p: (min(len(p), depth), p))
    n = len(pats)
    nb = min(nb, n)
    cost = {}
    for i in range(n):
        for j in range(i + 1, n + 1):
            cost[(i, j)] = bucket_cost(pats[i:j], depth)
    best = [[1e300] * (n + 1) for _ in range(nb + 1)]
    frm = [[0] * (n + 1) for _ in range(nb + 1)]
    best[0][0] = 0.0
    for k in range(1, nb + 1):
        for j in range(n + 1):
            for i in range(k - 1, j):
                if best[k - 1][i] < 1e300:
                    c = best[k - 1][i] + cost[(i, j)]
                    if c < best[k][j]:
                        best[k][j] = c
                        frm[k][j] = i
    cuts = [n]
    j = n
    for k in range(nb, 0, -1):
        j = frm[k][j]
        cuts.append(j)
    cuts = cuts[::-1]
    bucket = [0] * n
    for b in range(nb):
        for i in range(cuts[b], cuts[b + 1]):
            bucket[i] = b

    def total():
        return sum(bucket_cost([pats[i] for i in range(n) if bucket[i] == b], depth) for b in range(nb))
    cur = total()
    improved = True
    sweeps = 0
    while improved and sweeps < 30:
        improved = False
        sweeps += 1
        for i in range(n):
            a = bucket[i]
            bestc, to = cur, a
            for b in range(nb):
                if b == a:
                    continue
                bucket[i] = b
                c = total()
                if c < bestc - 1e-15:
                    bestc, to = c, b
            bucket[i] = to
            if to != a:
                cur = bestc
                improved = True
        for i in range(n):
            for j in range(i + 1, n):
                if bucket[i] == bucket[j]:
                    continue
                bucket[i], bucket[j] = bucket[j], bucket[i]
                c = total()
                if c < cur - 1e-15:
                    cur = c
                    improved = True
                else:
                    bucket[i], bucket[j] = bucket[j], bucket[i]
    return pats, bucket, cur


def stage_tables(pats, bucket, depth, nb):
    """A[d][byte] = bitmask of buckets passing byte at depth d"""
    A = np.zeros((depth, 256), dtype=np.uint32)
    for b in range(nb):
        mem = [p for p, bb in zip(pats, bucket) if bb == b]
        if not mem:
            continue
        for d in range(depth):
            if any(len(p) <= d for p in mem):
                A[d, :] |= 1 << b
            else:
                for p in mem:
                    A[d, p[d]] |= 1 << b
    return A


def rates(text, A, depth):
    n = len(text) - depth
    c = A[0][text[:n]]
    for d in range(1, depth):
        c = c & A[d][text[d:d + n]]
    cand = c != 0
    nul = text[:n] == 0
    rep = cand | nul
    g = n // 32 * 32
    groups = rep[:g].reshape(-1, 32).any(axis=1)
    quarters = rep[:g].reshape(-1, 8).any(axis=1)
    kb = g / 1024.0
    return cand[:g].sum() / kb, nul[:g].sum() / kb, groups.sum() / kb, quarters.sum() / kb


def main():
    pats = M.load_patterns(os.path.join(os.path.dirname(__file__), "..", "tests", "golden", "data", "strings.txt"))
    pats = [bytes(p) for p in pats]
    syn = M.Synth(seed=0xB200, payload_len=1400, len_mode=0, plants=2, plant_patterns=pats)
    data, offsets = syn.fill_host(0, 20000)
    text = np.frombuffer(data, dtype=np.uint8)[: int(offsets[-1])]
    rnd = np.random.default_rng(1).integers(0x20, 0x7f, size=len(text), dtype=np.uint8)
    print("C3 text: %d bytes; columns: candidates/KB, NULs/KB, 32-byte groups with a report/KB, 8-byte quarters/KB" % len(text))
    for depth, nb in [(4, 7), (4, 5), (3, 7), (3, 8), (4, 8), (3, 5), (2, 7), (4, 15), (3, 15)]:
        sp, bucket, est = optimise(pats, depth, nb)
        A = stage_tables(sp, bucket, depth, nb)
        r = rates(text, A, depth)
        r2 = rates(rnd, A, depth)
        print("depth %d buckets %2d: estimate %.2e/byte | C3 cand %.2f nul %.2f groups %.2f quarters %.2f | plain printable cand %.2f groups %.2f"
              % (depth, nb, est, r[0], r[1], r[2], r[3], r2[0], r2[2]))


if __name__ == "__main__" and len(sys.argv) == 1:
    main()


def main2():
    """geometries with the two-byte patterns in a chain of their own (exact pairs)"""
    pats = M.load_patterns(os.path.join(os.path.dirname(__file__), "..", "tests", "golden", "data", "strings.txt"))
    pats = [bytes(p) for p in pats]
    syn = M.Synth(seed=0xB200, payload_len=1400, len_mode=0, plants=2, plant_patterns=pats)
    data, offsets = syn.fill_host(0, 20000)
    text = np.frombuffer(data, dtype=np.uint8)[: int(offsets[-1])]
    short = sorted({p for p in pats if len(p) <= 2})
    longer = [p for p in pats if len(p) > 2]
    for depth, nb in [(4, 5), (4, 6), (3, 7), (4, 7)]:
        sp, bucket, est = optimise(longer, depth, nb)
        A = stage_tables(sp, bucket, depth, nb)
        # the short chain: bucket bit nb, exact in two bytes, open beyond
        for d in range(depth):
            if d >= 2:
                A[d, :] |= 1 << nb
            else:
                for p in short:
                    if len(p) > d:
                        A[d, p[d]] |= 1 << nb
                    else:
                        A[d, :] |= 1 << nb
        r = rates(text, A, depth)
        print("depth %d buckets %d (+ pair chain): C3 cand %.2f groups %.2f quarters %.2f" % (depth, nb, r[0], r[2], r[3]))


if __name__ == "__main__" and len(sys.argv) > 1 and sys.argv[1] == "2":
    main2()


GATE_MUL = 0x79B10000


def gate_table(pats):
    """automaton.c build_gate: (words, shift), or None when the gate would be too full to be built"""
    u = sorted(set(pats))
    keys = 256 * sum(len(p) == 1 for p in u) + len({p[:2] for p in u if len(p) >= 2})
    log_w = 5
    while (1 << log_w) < 1024 and (1 << log_w) < 16 * keys:
        log_w += 1
    shift = 32 - log_w
    g = np.zeros(1 << log_w, dtype=np.uint64)
    slot = lambda x: ((x * GATE_MUL) & 0xFFFFFFFF) >> shift
    for p in u:
        if len(p) == 1:
            for c in range(256):
                g[slot(p[0] | c << 8)] = 0xFFFFFFFF
        else:
            g[slot(p[0] | p[1] << 8)] |= 0xFFFFFFFF if len(p) == 2 else 0x80000000 >> (p[2] & 31)
    if 8 * sum(bin(int(w)).count("1") for w in g) > 32 * len(g):
        return None
    return g.astype(np.uint32), shift


def gate_model(text, A, depth, pats, gate):
    """per KB: events, candidates of the filter re-run / of the gate on the reported quarters / of both, true starts;
    verification rounds per resolve step (32 events, rounds of 32 candidates) = candidates per event"""
    words, shift = gate
    n = (len(text) - 40) // 32 * 32
    t = text.astype(np.uint32)
    c = A[0][text[:n]]
    for d in range(1, depth):
        c = c & A[d][text[d:d + n]]
    cand = (c != 0).reshape(-1, 32)
    nul = (text[:n] == 0).reshape(-1, 32)
    rep = cand | nul
    # the row loop's quarters: starts 0..8, 9..16, 17..24, 25..31; the gate tests those of each quarter that reported
    qrep = np.stack([rep[:, 0:9].any(1), rep[:, 9:17].any(1), rep[:, 17:25].any(1), rep[:, 25:32].any(1)], 1)
    win = np.zeros_like(cand)
    for k in range(4):
        win[:, (8 * k + 1 if k else 0):min(8 * k + 9, 32)] |= qrep[:, k:k + 1]
    key = t[:n] | t[1:n + 1] << 8
    slot = ((key.astype(np.uint64) * GATE_MUL) & 0xFFFFFFFF) >> shift
    gate_ok = ((words[slot.astype(np.int64)] >> (31 - (t[2:n + 2] & 31))) & 1).astype(bool).reshape(-1, 32)
    kb = n / 1024.0
    ev = rep.any(1).sum()
    now = (cand & win).sum()
    alone = (gate_ok & win).sum()
    both = (gate_ok & cand & win).sum()
    import re
    rx = re.compile(b"(?=(" + b"|".join(re.escape(p) for p in sorted(set(pats), key=len, reverse=True)) + b"))")
    true = len({m.start() for m in rx.finditer(text[:n].tobytes())})
    return dict(events=ev / kb, cand_rerun=now / kb, cand_gate=alone / kb, cand_both=both / kb, true_starts=true / kb,
                rounds_rerun=now / ev, rounds_gate=alone / ev, rounds_both=both / ev)


def main_gate(packets=8000):
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, root)
    import bench
    pats = [bytes(p) for p in M.load_patterns(os.path.join(root, "tests", "golden", "data", "strings.txt"))]
    data, offsets = bench.synth_stream(0xB200, 0, packets, 1400, 2, pats)
    text = np.frombuffer(bytes(data), dtype=np.uint8)
    sp, bucket, _ = optimise(pats, 4, 5)
    A = stage_tables(sp, bucket, 4, 5)
    g = gate_table(pats)
    print("gate: %d words, shift %d" % (len(g[0]), g[1]))
    r = gate_model(text, A, 4, pats, g)
    print("C3 (%d packets), per KB: events %.2f | candidates: filter re-run %.2f, gate %.2f, both %.2f, true starts %.2f"
          % (packets, r["events"], r["cand_rerun"], r["cand_gate"], r["cand_both"], r["true_starts"]))
    print("verification rounds per resolve step: filter re-run %.3f, gate %.3f, both %.3f"
          % (r["rounds_rerun"], r["rounds_gate"], r["rounds_both"]))


if __name__ == "__main__" and len(sys.argv) > 1 and sys.argv[1] == "gate":
    main_gate()
