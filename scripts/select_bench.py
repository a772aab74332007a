"""What selecting costs next to counting and finding, on bench.py's C3 workload (10 M x 1400-byte synthetic payloads
generated on the device, strings.txt, the same seed and plants), with the verdicts checked at full size.

Timed with CUDA events, warm-up first, the forms alternating within one process:
  count         kmpb_count_device_span (the count kernel, fused expansion)
  select        kmpb_select_device_span, verdicts only: the mark kernel (counts added too), the verdict pass
  select_index  the same with the index list: + the compaction (CUB DeviceSelect over the packet indices)
  find          kmpb_find_device_span unsorted: the find kernel, then the locate pass
The mark kernel and the verdict pass together are the profile bracket of a select call (kmpb_set_profile); the count
kernel alone that of a count call.  A separate pass after the timed rounds runs a few calls of each form under
torch.profiler (CUDA activities) and reports the device time per kernel name: where a select call's time goes between
the mark kernel, the verdict pass and the compaction.

Checks: the verdicts equal the set of packets that hold an (unsorted) find record, the index list is the flagged
packets in ascending order, the selected count matches it, and the counts a select call adds are the count call's.
Usage: python scripts/select_bench.py --out DIR [--packets N] [--rounds R] [--warmup W]
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

import multithreading_string_matching_b200 as kmp  # noqa: E402
from find_bench import SEED, card  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for select_bench.json")
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
    d_rec = torch.empty(total * 16, dtype=torch.uint8, device=dev)
    d_found = torch.zeros(1, dtype=torch.int64, device=dev)
    d_flags = torch.empty(n, dtype=torch.uint8, device=dev)
    d_flags2 = torch.empty(n, dtype=torch.uint8, device=dev)
    d_index = torch.empty(n, dtype=torch.int64, device=dev)
    d_sel = torch.zeros(1, dtype=torch.int64, device=dev)
    d_sel_counts = torch.zeros(len(patterns), dtype=torch.int64, device=dev)
    stream = torch.cuda.current_stream().cuda_stream

    def run(form):
        if form == "count":
            d_counts.zero_()
            m.count_device(d_bytes.data_ptr(), d_off.data_ptr(), n, d_counts.data_ptr(), span=span, stream=stream)
        elif form == "select":
            m.select_device(d_bytes.data_ptr(), d_off.data_ptr(), n, d_flags.data_ptr(), span, stream=stream)
        elif form == "select_index":
            d_sel_counts.zero_()
            m.select_device(d_bytes.data_ptr(), d_off.data_ptr(), n, d_flags2.data_ptr(), span, d_index.data_ptr(),
                            d_sel.data_ptr(), d_sel_counts.data_ptr(), stream=stream)
        else:
            m.find_device(d_bytes.data_ptr(), d_off.data_ptr(), n, d_rec.data_ptr(), total, d_found.data_ptr(), span,
                          stream=stream)

    forms = ["count", "select", "select_index", "find"]
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

    # ---- per-kernel device time, in a profiled pass of its own ----
    from torch.profiler import ProfilerActivity, profile

    prof_calls = 5
    per_kernel = {}
    for f in forms:
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(prof_calls):
                run(f)
            torch.cuda.synchronize()
        rows = {}
        for e in prof.key_averages():
            t = getattr(e, "self_device_time_total", None)
            if t is None:
                t = e.self_cuda_time_total
            if t > 0:
                rows[e.key[:80]] = round(t / 1000.0 / prof_calls, 4)  # ms per call
        per_kernel[f] = dict(sorted(rows.items(), key=lambda kv: -kv[1]))

    # ---- checks ----
    t0 = time.time()
    assert int(d_found.item()) == total
    pk = np.unique(d_rec.cpu().numpy().view(kmp.MATCH_DTYPE)["packet"].astype(np.int64))
    flags = d_flags.cpu().numpy().astype(bool)
    want = np.zeros(n, dtype=bool)
    want[pk] = True
    n_sel = int(d_sel.item())
    med = {f: float(np.median(times[f])) for f in forms}
    result = {
        "workload": "C3: %d x %d B synthetic payloads (seed 0x%X, 2 plants per packet), strings.txt (%d patterns)"
                    % (n, L, SEED, len(patterns)),
        "card": card(),
        "rounds": args.rounds, "warmup": args.warmup,
        "matches": total,
        "selected_packets": n_sel,
        "ms": {f: {"median": med[f], "min": float(np.min(times[f])), "max": float(np.max(times[f]))} for f in forms},
        "kernel_ms": {f: float(np.median(kernel[f])) for f in forms},
        "profiled_ms_per_call_by_kernel": per_kernel,
        "select_over_count": med["select"] / med["count"],
        "select_index_over_count": med["select_index"] / med["count"],
        "find_over_count": med["find"] / med["count"],
        "bitmap_bytes": (nbytes + 31) // 32 * 4,
        "payload_bytes": nbytes,
        "checks": {"flags_are_the_packets_of_find_records": bool(np.array_equal(flags, want)),
                   "index_is_flatnonzero": bool(np.array_equal(d_index[:n_sel].cpu().numpy(), pk)),
                   "both_selects_agree": bool(np.array_equal(d_flags2.cpu().numpy().astype(bool), flags)),
                   "select_counts_are_the_counts": bool(np.array_equal(d_sel_counts.cpu().numpy(), counts))},
        "check_seconds": round(time.time() - t0, 1),
    }
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "select_bench.json"), "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result))
    sys.exit(0 if all(result["checks"].values()) else 1)


if __name__ == "__main__":
    main()
