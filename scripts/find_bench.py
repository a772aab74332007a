"""What finding costs next to counting, on bench.py's C3 workload (10 M x 1400-byte synthetic payloads generated on the
device, strings.txt, the same seed and plants), with the records checked at full size without an oracle.

Timed with CUDA events, warm-up first, the forms alternating within one process:
  count       kmpb_count_device_span (the count kernel, fused expansion)
  find        kmpb_find_device_span unsorted: the find kernel, then the locate pass
  find_sorted kmpb_find_device_span with KMPB_FIND_SORTED: find kernel, sort keys, radix sort, locate
  find_cap0   kmpb_find_device_span with capacity 0: the find kernel reserves slots and counts, writes no record (what
              the reservation atomics cost without the record traffic)
The find kernel's own time comes from the profile events around it (kmpb_set_profile), the rest of a find call is the
locate (and sort) work.

Checks on the sorted records (the unsorted ones must be a permutation of them):
  validity     payload[packet][offset : offset + len] == pattern, offset + len <= packet length, no NUL before the end
  distinctness strictly increasing (packet, offset, pattern): sorted and no duplicates
  cardinality  the per-pattern histogram equals the count vector (and the count vector sums to the known total)
Usage: python scripts/find_bench.py --out DIR [--packets N] [--rounds R] [--warmup W]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import multithreading_string_matching_b200 as kmp  # noqa: E402

SEED = 0xB200           # bench.py's
C3_COUNT_SUM = 33_812_242  # sum of the count vector of the default 10 M-packet stream (duplicate tokens counted each time)


def card():
    import torch

    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["max_sm_clock"] = [v.strip() for v in q.split(",")]
    except Exception as e:  # the number is still worth having; say why the card's settings are missing
        info["power_limit"] = "unknown (%s)" % e
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for find_bench.json")
    ap.add_argument("--packets", type=int, default=10_000_000)
    ap.add_argument("--rounds", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    import torch

    dev = "cuda:0"
    L, n = 1400, args.packets
    patterns = kmp.load_patterns(os.path.join(ROOT, "tests", "golden", "data", "strings.txt"))
    m = kmp.Matcher(0)
    m.set_patterns(patterns)
    synth = kmp.Synth(seed=SEED, payload_len=L, plants=2, plant_patterns=patterns)
    nbytes = synth.nbytes(0, n)
    d_bytes = torch.empty(nbytes + 4096, dtype=torch.uint8, device=dev)
    d_bytes[nbytes:].zero_()
    d_off = torch.empty(n + 1, dtype=torch.int64, device=dev)
    synth.fill_device(m, 0, n, d_bytes.data_ptr(), d_off.data_ptr())
    span = (0, nbytes)
    d_counts = torch.zeros(len(patterns), dtype=torch.int64, device=dev)
    m.count_device(d_bytes.data_ptr(), d_off.data_ptr(), n, d_counts.data_ptr(), span=span)
    torch.cuda.synchronize()
    counts = d_counts.cpu().numpy()
    firsts, seen = [], {}
    for i, p in enumerate(patterns):
        firsts.append(seen.setdefault(p, i))
    total = int(sum(counts[i] for i in range(len(patterns)) if firsts[i] == i))
    cap = total
    d_out = torch.empty(cap * 16, dtype=torch.uint8, device=dev)
    d_out2 = torch.empty(cap * 16, dtype=torch.uint8, device=dev)
    d_n = torch.zeros(1, dtype=torch.int64, device=dev)
    stream = torch.cuda.current_stream().cuda_stream

    def run(form):
        if form == "find_cap0":
            m.find_device(d_bytes.data_ptr(), d_off.data_ptr(), n, 0, 0, d_n.data_ptr(), span, stream=stream)
        elif form == "count":
            d_counts.zero_()
            m.count_device(d_bytes.data_ptr(), d_off.data_ptr(), n, d_counts.data_ptr(), span=span, stream=stream)
        else:
            out = d_out if form == "find_sorted" else d_out2
            m.find_device(d_bytes.data_ptr(), d_off.data_ptr(), n, out.data_ptr(), cap, d_n.data_ptr(), span,
                          sorted=form == "find_sorted", stream=stream)

    forms = ["count", "find", "find_sorted", "find_cap0"]
    m.set_profile(True)
    times = {f: [] for f in forms}
    kernel = {f: [] for f in forms}
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    for r in range(args.warmup + args.rounds):
        for f in forms:
            ev[0].record()
            run(f)
            ev[1].record()
            torch.cuda.synchronize()
            if r >= args.warmup:
                times[f].append(ev[0].elapsed_time(ev[1]))
                kernel[f].append(m.last_kernel_ms())
    m.set_profile(False)
    assert int(d_n.item()) == total

    # ---- checks ----
    t0 = time.time()
    rec = d_out.cpu().numpy().view(kmp.MATCH_DTYPE)
    unsorted = d_out2.cpu().numpy().view(kmp.MATCH_DTYPE)
    pk, of, pt = rec["packet"].astype(np.int64), rec["offset"].astype(np.int64), rec["pattern"].astype(np.int64)
    key_increasing = (np.diff(pk) > 0) | ((np.diff(pk) == 0) & ((np.diff(of) > 0) | ((np.diff(of) == 0) & (np.diff(pt) > 0))))
    distinct_sorted = bool(key_increasing.all())
    permutation = bool(np.array_equal(np.sort(unsorted, order=["packet", "offset", "pattern"]), rec))
    hist = np.bincount(pt, minlength=len(patterns))
    cardinality = bool(all(int(hist[firsts[i]]) == int(counts[i]) for i in range(len(patterns))))
    lens = np.array([len(p) for p in patterns], dtype=np.int64)
    maxlen = int(lens.max())
    table = np.zeros((len(patterns), maxlen), dtype=np.uint8)
    for i, p in enumerate(patterns):
        table[i, : len(p)] = np.frombuffer(p, dtype=np.uint8)
    off_h = d_off.cpu().numpy()
    plen = off_h[pk + 1] - off_h[pk]
    mlen = lens[pt]
    # first NUL of every packet (every C3 payload ends with one), on the device
    first_nul = (d_bytes[:nbytes].view(n, L) == 0).to(torch.uint8).argmax(dim=1).cpu().numpy().astype(np.int64)
    valid = (of + mlen <= plen) & (of + mlen <= first_nul[pk])
    d_pos = torch.from_numpy(off_h[pk] + of).to(dev)
    ar = torch.arange(maxlen, device=dev)
    same = np.empty(len(rec), dtype=bool)
    step = 4_000_000
    for a in range(0, len(rec), step):
        idx = (d_pos[a:a + step, None] + ar[None, :]).clamp_(max=nbytes + 4095)
        window = d_bytes[idx].cpu().numpy()
        mask = np.arange(maxlen)[None, :] < mlen[a:a + step, None]
        same[a:a + step] = ((window == table[pt[a:a + step]]) | ~mask).all(axis=1)
    valid &= same
    result = {
        "workload": "C3: %d x %d B synthetic payloads (seed 0x%X, 2 plants per packet), strings.txt (%d patterns)"
                    % (n, L, SEED, len(patterns)),
        "card": card(),
        "rounds": args.rounds, "warmup": args.warmup,
        "matches": total,
        "count_sum": int(counts.sum()),
        "ms": {f: {"median": float(np.median(times[f])), "min": float(np.min(times[f])), "max": float(np.max(times[f]))}
               for f in forms},
        "kernel_ms": {f: float(np.median(kernel[f])) for f in forms},
        "find_over_count": float(np.median(times["find"]) / np.median(times["count"])),
        "find_sorted_over_count": float(np.median(times["find_sorted"]) / np.median(times["count"])),
        "record_bytes": total * 16,
        "payload_bytes": nbytes,
        "checks": {"valid": bool(valid.all()), "invalid_records": int((~valid).sum()), "distinct_and_sorted": distinct_sorted,
                   "unsorted_is_a_permutation": permutation, "cardinality": cardinality,
                   "count_sum_is_known": int(counts.sum()) == C3_COUNT_SUM if n == 10_000_000 else None},
        "check_seconds": round(time.time() - t0, 1),
    }
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "find_bench.json"), "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result))
    ok = all(v is not False for k, v in result["checks"].items() if k != "invalid_records")
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
