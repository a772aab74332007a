"""What position windows cost, on bench.py's C3 workload (10 M x 1400-byte synthetic payloads generated on the device,
strings.txt, the same seed and plants), device-resident, with every answer checked.

Sets, each on a context of its own, timed with CUDA events in alternating rounds after a warm-up (medians):
  ref       strings.txt without windows: the reference time (and the unwindowed twin of `all64`)
  plus16    strings.txt plus 16 windowed patterns, strings.txt tokens (C3 plants them, so they match) with window
            [0, 128 - len]: every window ends by byte 128 of the payload; the union kernel's set is ref's
  all64     every strings.txt token windowed [0, 64]: the union kernel does not run, the window kernel reads 65..163
            bytes of each 1400-byte payload
plus, for plus16, a find call (unsorted, exact capacity) and a select call (verdicts only).  With --parent-lib, the
`ref` count call of another build of libkmpb200.so (e.g. the parent commit's) joins the alternation as `ref_parent`,
through the C ABI on the same device buffers, to show that the unwindowed count path is unchanged.  The profile bracket
(kmpb_set_profile) of each count call gives its kernels' time.

Checks: each set's counts equal the per-pattern engine's on the full batch, and on a 20 000-packet slice made on the
host the union engine's counts and find records equal the reference finder's (tests/c/kmp_find_ref.c) filtered by the
windows; plus16's find records and verdicts agree with its counts.
Usage: python scripts/window_bench.py --out DIR [--packets N] [--rounds R] [--warmup W] [--parent-lib PATH]
"""
import argparse
import ctypes
import json
import os
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

import multithreading_string_matching_b200 as kmp  # noqa: E402
from find_bench import SEED, card  # noqa: E402


def sets(tokens):
    distinct = sorted(set(tokens), key=tokens.index)
    extra = [t for t in distinct if len(t) <= 40][:16]
    return {
        "ref": (tokens, None),
        "plus16": (tokens + extra, [None] * len(tokens) + [(0, 128 - len(t)) for t in extra]),
        "all64": (tokens, (0, 64)),
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for r07_window_c3.json")
    ap.add_argument("--packets", type=int, default=10_000_000)
    ap.add_argument("--rounds", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--parent-lib", help="another libkmpb200.so whose unwindowed count call is timed beside ours")
    args = ap.parse_args()
    import torch
    from test_find import RefFinder
    from test_windows import expected

    dev = "cuda:0"
    L, n = 1400, args.packets
    tokens = kmp.load_patterns(os.path.join(ROOT, "tests", "golden", "data", "strings.txt"))
    cases = sets(tokens)
    ms = {}
    for name, (pats, win) in cases.items():
        ms[name] = kmp.Matcher(0)
        ms[name].set_patterns(pats, window=win)
    synth = kmp.Synth(seed=SEED, payload_len=L, plants=2, plant_patterns=tokens)
    nbytes = synth.nbytes(0, n)
    d_bytes = torch.empty(nbytes + 4096, dtype=torch.uint8, device=dev)
    d_bytes[nbytes:].zero_()
    d_off = torch.empty(n + 1, dtype=torch.int64, device=dev)
    synth.fill_device(ms["ref"], 0, n, d_bytes.data_ptr(), d_off.data_ptr())
    span = (0, nbytes)
    stream = torch.cuda.current_stream().cuda_stream
    d_counts = {k: torch.zeros(len(p), dtype=torch.int64, device=dev) for k, (p, _) in cases.items()}

    def count(name):
        d_counts[name].zero_()
        ms[name].count_device(d_bytes.data_ptr(), d_off.data_ptr(), n, d_counts[name].data_ptr(), span=span, stream=stream)

    for name in cases:
        count(name)
    torch.cuda.synchronize()
    counts = {k: d_counts[k].cpu().tolist() for k in cases}
    p16, w16 = cases["plus16"]
    seen = {}
    firsts = [seen.setdefault((p, w), i) for i, (p, w) in enumerate(zip(p16, w16))]
    total16 = sum(counts["plus16"][i] for i in range(len(p16)) if firsts[i] == i)
    d_rec = torch.empty(total16 * 16, dtype=torch.uint8, device=dev)
    d_found = torch.zeros(1, dtype=torch.int64, device=dev)
    d_flags = torch.empty(n, dtype=torch.uint8, device=dev)

    def find():
        ms["plus16"].find_device(d_bytes.data_ptr(), d_off.data_ptr(), n, d_rec.data_ptr(), total16, d_found.data_ptr(),
                                 span, stream=stream)

    def select():
        ms["plus16"].select_device(d_bytes.data_ptr(), d_off.data_ptr(), n, d_flags.data_ptr(), span, stream=stream)

    forms = {"ref": lambda: count("ref"), "plus16": lambda: count("plus16"), "all64": lambda: count("all64"),
             "plus16_find": find, "plus16_select": select}
    if args.parent_lib:
        P = ctypes.CDLL(os.path.abspath(args.parent_lib))
        vp, u64 = ctypes.c_void_p, ctypes.c_uint64
        P.kmpb_create.argtypes = [ctypes.POINTER(vp), ctypes.c_int]
        P.kmpb_set_patterns.argtypes = [vp, vp, vp, ctypes.c_uint32]
        P.kmpb_count_device_span.argtypes = [vp, vp, vp, u64, u64, u64, vp, vp]
        P.kmpb_set_profile.argtypes = [vp, ctypes.c_int]
        P.kmpb_last_kernel_ms.argtypes = [vp, ctypes.POINTER(ctypes.c_double)]
        pctx = vp()
        blob, off = kmp.pack_patterns(tokens)
        assert P.kmpb_create(ctypes.byref(pctx), 0) == 0 and P.kmpb_set_patterns(pctx, blob.ctypes.data, off.ctypes.data, len(tokens)) == 0
        P.kmpb_set_profile(pctx, 1)
        d_parent = torch.zeros(len(tokens), dtype=torch.int64, device=dev)

        def ref_parent():
            d_parent.zero_()
            assert P.kmpb_count_device_span(pctx, d_bytes.data_ptr(), d_off.data_ptr(), n, 0, nbytes, d_parent.data_ptr(),
                                            stream) == 0

        def parent_kernel_ms():
            v = ctypes.c_double()
            assert P.kmpb_last_kernel_ms(pctx, ctypes.byref(v)) == 0
            return v.value

        forms["ref_parent"] = ref_parent
    for m in ms.values():
        m.set_profile(True)
    times = {f: [] for f in forms}
    kernel = {f: [] for f in forms}
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    for r in range(args.warmup + args.rounds):
        for f, run in forms.items():
            ev[0].record()
            run()
            ev[1].record()
            torch.cuda.synchronize()
            if r >= args.warmup:
                times[f].append(ev[0].elapsed_time(ev[1]))
                kernel[f].append(parent_kernel_ms() if f == "ref_parent" else ms[f.split("_")[0]].last_kernel_ms())

    # ---- checks: the per-pattern engine on the full batch, the reference finder on a host slice ----
    checks = {}
    if args.parent_lib:
        checks["ref_parent_counts_equal_ours"] = d_parent.cpu().tolist() == counts["ref"]
    for name, (pats, win) in cases.items():
        with kmp.Matcher(0, engine="perpat") as pp:
            pp.set_patterns(pats, window=win)
            c = torch.zeros(len(pats), dtype=torch.int64, device=dev)
            pp.count_device(d_bytes.data_ptr(), d_off.data_ptr(), n, c.data_ptr(), span=span)
            torch.cuda.synchronize()
            checks[name + "_counts_equal_the_perpat_engine"] = c.cpu().tolist() == counts[name]
    rec = d_rec.cpu().numpy()[: 16 * total16].view(kmp.MATCH_DTYPE)
    checks["plus16_find_total_is_the_counts"] = int(d_found.item()) == total16
    verdicts = np.zeros(n, dtype=bool)
    verdicts[rec["packet"].astype(np.int64)] = True
    checks["plus16_verdicts_are_the_packets_of_find_records"] = bool(np.array_equal(d_flags.cpu().numpy().astype(bool), verdicts))
    k = 20_000
    data, offsets = synth.fill_host(0, k)
    with tempfile.TemporaryDirectory() as tmp:
        finder = RefFinder(tmp)
        for name, (pats, win) in cases.items():
            want_counts, want, _ = expected(finder, pats, False, win if win is not None else [None] * len(pats), data, offsets)
            checks[name + "_slice_counts_equal_the_reference"] = ms[name].count_host(data, offsets) == want_counts
            checks[name + "_slice_records_equal_the_reference"] = bool(np.array_equal(ms[name].find_host(data, offsets), want))

    med = {f: float(np.median(times[f])) for f in forms}
    result = {
        "workload": "C3: %d x %d B synthetic payloads (seed 0x%X, 2 plants per packet), device-resident" % (n, L, SEED),
        "card": card(),
        "rounds": args.rounds, "warmup": args.warmup,
        "sets": {"ref": "strings.txt (%d patterns), no windows" % len(tokens),
                 "plus16": "strings.txt + 16 windowed tokens, window [0, 128 - len]",
                 "all64": "every strings.txt token windowed [0, 64]"},
        "matches": {k: int(sum(v)) for k, v in counts.items()},
        "ms": {f: {"median": med[f], "min": float(np.min(times[f])), "max": float(np.max(times[f]))} for f in forms},
        "kernel_ms": {f: float(np.median(kernel[f])) for f in forms},
        "plus16_over_ref": med["plus16"] / med["ref"],
        "all64_over_ref": med["all64"] / med["ref"],
        "plus16_find_over_ref": med["plus16_find"] / med["ref"],
        "plus16_select_over_ref": med["plus16_select"] / med["ref"],
        "ref_over_ref_parent": med["ref"] / med["ref_parent"] if args.parent_lib else None,
        "targets": {"plus16_over_ref": 1.25, "all64_over_ref": 0.35},
        "payload_bytes": nbytes,
        "checks": checks,
    }
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "r07_window_c3.json"), "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result))
    sys.exit(0 if all(checks.values()) else 1)


if __name__ == "__main__":
    main()
