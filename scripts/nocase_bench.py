"""What case-insensitive patterns cost, on bench.py's C3 workload (10 M x 1400-byte synthetic payloads generated on the
device, seed 0xB200, strings.txt), with find_bench.py's conventions: CUDA events, warm-up first, the forms alternating
within one process, the card's name and power limit read in the same run.  One context per form:
  plain    strings.txt through kmpb_set_patterns
  zero     the same through kmpb_set_patterns_ex with all-zero flags (the same tables, the same kernels)
  nocase   every token KMPB_PAT_NOCASE (the nocase kernels)
For each: the count call (kmpb_count_device_span) and its kernel (profile events), and the unsorted find call.

Checks:
  count_sum_is_known      the case-sensitive count vector sums to the known C3 total, in both case-sensitive forms
  zero_equals_plain       the two case-sensitive count vectors are equal
  nocase_at_least         every nocase count >= its case-sensitive count, equal for tokens without letters
  valid / distinct_and_sorted / cardinality
                          find_bench.py's checks on the sorted nocase records, validity compared after folding
  oracle_200k             on the first 200 k packets the nocase counts equal the oracle's on the folded copy
Usage: python scripts/nocase_bench.py --out DIR [--packets N] [--rounds R] [--warmup W]
"""
import argparse
import ctypes
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import multithreading_string_matching_b200 as kmp  # noqa: E402
from find_bench import C3_COUNT_SUM, SEED, card  # noqa: E402

LETTERS = set(range(0x41, 0x5B)) | set(range(0x61, 0x7B))


def fold_np(a):
    a = a.copy()
    up = (a >= 0x41) & (a <= 0x5A)
    a[up] += 32
    return a


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for nocase_bench.json")
    ap.add_argument("--packets", type=int, default=10_000_000)
    ap.add_argument("--rounds", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    import torch

    from oracle import oracle_py

    dev = "cuda:0"
    L, n = 1400, args.packets
    patterns = kmp.load_patterns(os.path.join(ROOT, "tests", "golden", "data", "strings.txt"))
    P = len(patterns)
    blob, off = kmp.pack_patterns(patterns)
    u8p, u32p = ctypes.POINTER(ctypes.c_uint8), ctypes.POINTER(ctypes.c_uint32)
    forms = ["plain", "zero", "nocase"]
    ms = {f: kmp.Matcher(0) for f in forms}
    kmp._lib.check(kmp.lib().kmpb_set_patterns(ms["plain"].handle, blob.ctypes.data_as(u8p), off.ctypes.data_as(u32p), P))
    zeros = np.zeros(P, dtype=np.uint8)
    kmp._lib.check(kmp.lib().kmpb_set_patterns_ex(ms["zero"].handle, blob.ctypes.data_as(u8p), off.ctypes.data_as(u32p), P,
                                                  zeros.ctypes.data_as(u8p)))
    ms["nocase"].set_patterns(patterns, nocase=True)
    for f in ("plain", "zero"):  # Matcher.set_patterns was bypassed: the count helpers need the pattern list
        ms[f].patterns = list(patterns)

    synth = kmp.Synth(seed=SEED, payload_len=L, plants=2, plant_patterns=patterns)
    nbytes = synth.nbytes(0, n)
    d_bytes = torch.empty(nbytes + 4096, dtype=torch.uint8, device=dev)
    d_bytes[nbytes:].zero_()
    d_off = torch.empty(n + 1, dtype=torch.int64, device=dev)
    synth.fill_device(ms["plain"], 0, n, d_bytes.data_ptr(), d_off.data_ptr())
    span = (0, nbytes)
    stream = torch.cuda.current_stream().cuda_stream
    d_counts = {f: torch.zeros(P, dtype=torch.int64, device=dev) for f in forms}
    for f in forms:
        ms[f].count_device(d_bytes.data_ptr(), d_off.data_ptr(), n, d_counts[f].data_ptr(), span=span, stream=stream)
    torch.cuda.synchronize()
    counts = {f: d_counts[f].cpu().numpy() for f in forms}
    firsts, seen, firsts_nc, seen_nc = [], {}, [], {}
    for i, p in enumerate(patterns):
        firsts.append(seen.setdefault(p, i))
        firsts_nc.append(seen_nc.setdefault(p.lower(), i))
    totals = {f: int(sum(counts[f][i] for i in range(P) if (firsts_nc if f == "nocase" else firsts)[i] == i)) for f in forms}
    cap = max(totals.values())
    d_out = torch.empty(cap * 16, dtype=torch.uint8, device=dev)
    d_n = torch.zeros(1, dtype=torch.int64, device=dev)

    times = {(f, k): [] for f in forms for k in ("count", "find")}
    kernel = {f: [] for f in forms}
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    for f in forms:
        ms[f].set_profile(True)
    for r in range(args.warmup + args.rounds):
        for f in forms:
            for k in ("count", "find"):
                ev[0].record()
                if k == "count":
                    d_counts[f].zero_()
                    ms[f].count_device(d_bytes.data_ptr(), d_off.data_ptr(), n, d_counts[f].data_ptr(), span=span, stream=stream)
                else:
                    ms[f].find_device(d_bytes.data_ptr(), d_off.data_ptr(), n, d_out.data_ptr(), cap, d_n.data_ptr(), span,
                                      stream=stream)
                ev[1].record()
                torch.cuda.synchronize()
                if k == "count" and r >= args.warmup:
                    kernel[f].append(ms[f].last_kernel_ms())
                if r >= args.warmup:
                    times[(f, k)].append(ev[0].elapsed_time(ev[1]))
                if k == "find":
                    assert int(d_n.item()) == totals[f], f
    for f in forms:
        ms[f].set_profile(False)

    # ---- checks ----
    t0 = time.time()
    cs, nc = counts["plain"], counts["nocase"]
    letterless = [not any(c in LETTERS for c in p) for p in patterns]
    nocase_at_least = bool(all(nc[i] >= cs[i] and (nc[i] == cs[i] or not letterless[i]) for i in range(P)))
    ms["nocase"].find_device(d_bytes.data_ptr(), d_off.data_ptr(), n, d_out.data_ptr(), cap, d_n.data_ptr(), span,
                             sorted=True, stream=stream)
    torch.cuda.synchronize()
    total = totals["nocase"]
    rec = d_out[: 16 * total].cpu().numpy().view(kmp.MATCH_DTYPE)
    pk, of, pt = rec["packet"].astype(np.int64), rec["offset"].astype(np.int64), rec["pattern"].astype(np.int64)
    key_increasing = (np.diff(pk) > 0) | ((np.diff(pk) == 0) & ((np.diff(of) > 0) | ((np.diff(of) == 0) & (np.diff(pt) > 0))))
    hist = np.bincount(pt, minlength=P)
    cardinality = bool(all(int(hist[firsts_nc[i]]) == int(nc[i]) for i in range(P)))
    lens = np.array([len(p) for p in patterns], dtype=np.int64)
    maxlen = int(lens.max())
    table = np.zeros((P, maxlen), dtype=np.uint8)
    for i, p in enumerate(patterns):
        table[i, : len(p)] = fold_np(np.frombuffer(p, dtype=np.uint8))
    off_h = d_off.cpu().numpy()
    plen = off_h[pk + 1] - off_h[pk]
    mlen = lens[pt]
    first_nul = (d_bytes[:nbytes].view(n, L) == 0).to(torch.uint8).argmax(dim=1).cpu().numpy().astype(np.int64)
    valid = (of + mlen <= plen) & (of + mlen <= first_nul[pk])
    d_pos = torch.from_numpy(off_h[pk] + of).to(dev)
    ar = torch.arange(maxlen, device=dev)
    same = np.empty(len(rec), dtype=bool)
    step = 4_000_000
    for a in range(0, len(rec), step):
        idx = (d_pos[a:a + step, None] + ar[None, :]).clamp_(max=nbytes + 4095)
        window = fold_np(d_bytes[idx].cpu().numpy())
        mask = np.arange(maxlen)[None, :] < mlen[a:a + step, None]
        same[a:a + step] = ((window == table[pt[a:a + step]]) | ~mask).all(axis=1)
    valid &= same
    # the oracle on the folded copy of the first 200 k packets
    n_o = min(n, 200_000)
    d_sub = torch.zeros(P, dtype=torch.int64, device=dev)
    ms["nocase"].count_device(d_bytes.data_ptr(), d_off.data_ptr(), n_o, d_sub.data_ptr(), span=(0, int(off_h[n_o])),
                              stream=stream)
    torch.cuda.synchronize()
    folded = fold_np(d_bytes[: int(off_h[n_o])].cpu().numpy())
    want = oracle_py.count_csr(folded, off_h[: n_o + 1].astype(np.uint64), [p.lower() for p in patterns])
    oracle_200k = d_sub.cpu().tolist() == want

    def stat(v):
        return {"median": float(np.median(v)), "min": float(np.min(v)), "max": float(np.max(v))}

    result = {
        "workload": "C3: %d x %d B synthetic payloads (seed 0x%X, 2 plants per packet), strings.txt (%d patterns)"
                    % (n, L, SEED, P),
        "card": card(),
        "rounds": args.rounds, "warmup": args.warmup,
        "forms": {"plain": "kmpb_set_patterns", "zero": "kmpb_set_patterns_ex, all-zero flags",
                  "nocase": "kmpb_set_patterns_ex, every token KMPB_PAT_NOCASE"},
        "count_ms": {f: stat(times[(f, "count")]) for f in forms},
        "kernel_ms": {f: stat(kernel[f]) for f in forms},
        "find_ms": {f: stat(times[(f, "find")]) for f in forms},
        "count_gbps": {f: nbytes / (np.median(times[(f, "count")]) * 1e-3) / 1e9 for f in forms},
        "nocase_over_plain": {"count": float(np.median(times[("nocase", "count")]) / np.median(times[("plain", "count")])),
                              "kernel": float(np.median(kernel["nocase"]) / np.median(kernel["plain"])),
                              "find": float(np.median(times[("nocase", "find")]) / np.median(times[("plain", "find")]))},
        "matches": totals,
        "count_sum": {f: int(counts[f].sum()) for f in forms},
        "payload_bytes": nbytes,
        "checks": {"count_sum_is_known": (int(cs.sum()) == C3_COUNT_SUM and int(counts["zero"].sum()) == C3_COUNT_SUM)
                   if n == 10_000_000 else None,
                   "zero_equals_plain": bool(np.array_equal(counts["zero"], cs)),
                   "nocase_at_least": nocase_at_least,
                   "valid": bool(valid.all()), "invalid_records": int((~valid).sum()),
                   "distinct_and_sorted": bool(key_increasing.all()), "cardinality": cardinality,
                   "oracle_200k": oracle_200k},
        "check_seconds": round(time.time() - t0, 1),
    }
    for m in ms.values():
        m.close()
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "nocase_bench.json"), "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result))
    ok = all(v is not False for k, v in result["checks"].items() if k != "invalid_records")
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
