#!/usr/bin/env python3
"""What the union kernel's resolve steps do on C3, counted on the GPU: events, resolve steps, candidates appended and
verification rounds, per KB of payload and per resolve step.  Builds the library with the diagnostic counters
(EXTRA_NVFLAGS=-DKMPB_UN_STATS, absent from the production build) into a temporary directory, so the tree is left as
it is.  scripts/filter_model.py gate models the same numbers on the CPU.
With --nocase every token of strings.txt is case-insensitive (KMPB_PAT_NOCASE).
Usage: scripts/event_counts.py [--packets N] [--flags "-DKMPB_UN_GATE_AND"] [--nocase]"""
import argparse, ctypes, json, os, shutil, subprocess, sys, tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = "multithreading_string_matching_b200"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--packets", type=int, default=2_000_000, help="C3 packets of 1400 bytes")
    ap.add_argument("--flags", default="", help="more nvcc flags for the diagnostic build")
    ap.add_argument("--nocase", action="store_true", help="every pattern case-insensitive")
    args = ap.parse_args()
    tmp = tempfile.mkdtemp(prefix="kmpb_stats_")
    try:
        shutil.copytree(os.path.join(ROOT, "include"), os.path.join(tmp, "include"))
        shutil.copytree(os.path.join(ROOT, PKG), os.path.join(tmp, PKG),
                        ignore=shutil.ignore_patterns("build", "bin", "*.so", "__pycache__"))
        subprocess.run(["make", "-s", "-j8", "-C", os.path.join(tmp, PKG),
                        "EXTRA_NVFLAGS=-DKMPB_UN_STATS " + args.flags], check=True, stdout=subprocess.DEVNULL)
        sys.path.insert(0, tmp)
        import torch
        import multithreading_string_matching_b200 as kmp
        from multithreading_string_matching_b200 import _lib
        assert os.path.dirname(kmp.__file__).startswith(tmp)
        L = _lib.lib()
        L.kmpb_union_stats.argtypes = [ctypes.POINTER(ctypes.c_uint64), ctypes.c_int]
        pats = kmp.load_patterns(os.path.join(ROOT, "tests", "golden", "data", "strings.txt"))
        m = kmp.Matcher(0, engine="union")
        m.set_patterns(pats, nocase=args.nocase)
        synth = kmp.Synth(seed=0xB200, payload_len=1400, plants=2, plant_patterns=pats)
        n = args.packets
        nb = synth.nbytes(0, n)
        d_bytes = torch.empty(nb + 4096, dtype=torch.uint8, device="cuda:0")
        d_bytes[nb:].zero_()
        d_off = torch.empty(n + 1, dtype=torch.int64, device="cuda:0")
        synth.fill_device(m, 0, n, d_bytes.data_ptr(), d_off.data_ptr())
        d_counts = torch.zeros(len(pats), dtype=torch.int64, device="cuda:0")
        st = (ctypes.c_uint64 * 4)()
        L.kmpb_union_stats(st, 1)
        m.count_device(d_bytes.data_ptr(), d_off.data_ptr(), n, d_counts.data_ptr(), span=(0, nb),
                       stream=torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        L.kmpb_union_stats(st, 1)
        ev, steps, cand, rounds = (int(x) for x in st)
        kb = nb / 1024.0
        print(json.dumps({"packets": n, "bytes": nb, "flags": args.flags, "nocase": args.nocase, "matches": int(d_counts.sum().item()),
                          "events": ev, "resolve_steps": steps, "candidates": cand, "verify_rounds": rounds,
                          "events_per_kb": round(ev / kb, 4), "candidates_per_kb": round(cand / kb, 4),
                          "candidates_per_event": round(cand / max(ev, 1), 4),
                          "verify_rounds_per_step": round(rounds / max(steps, 1), 4)}))
        m.close()
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


if __name__ == "__main__":
    main()
