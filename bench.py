#!/usr/bin/env python3
"""bench.py -- payload GB/s of the KMP packet-matching hot path on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (BASELINE.json configs[2]): synthetic UDP stream, 10 M packets x 1400-byte payloads per GPU
(counter-based generator, csrc/cuda/synth.cu; last payload byte NUL, 2 strings.txt tokens planted per
packet), matched against the 97 patterns of the bundled strings.txt.  Packets are split over ranks as
mpi_dumping.c:149-157 splits them; weak scaling: the stream grows with N, each GPU matches its own
contiguous slice and the 97-entry count vectors are summed with one NCCL all-reduce (mpi_dumping.c:202).

A "step" is one pass of the hot path over the rank's whole slice.
  value  device-resident: payload already in HBM when the timed region starts (CUDA events, max over ranks)
  e2e    the same pass through the C ABI's host entry point kmpb_count_host: pinned host CSR -> chunked
         H2D on 4 streams overlapped with the kernels -> counts back on the host
  roofline      the union kernel alone (events around the kernel on its stream) vs the measured HBM peak
  cpu_baseline  the unmodified reference on a bounded prefix of the same stream: oracle/_ref/openmp_data on all host
                threads, and under "serial" oracle/_ref/serial on one core (a shorter prefix) -- reported baselines,
                not the target
  parity_full   the per-pattern engine (kmpb_perpat_kernel) over every rank's whole slice == the union engine's counts
  strong        (N > 1) the fixed stream of ONE GPU's size split over the ranks as mpi_dumping.c:149-157 splits it
  sweep         small forms of BASELINE configs[3] (pattern sweep) and configs[4] (mixed payload sizes), each with its
                own parity check; the full forms: --config c4 | c5, and --config cli for bin/kmp_match on a large savefile
--impl reference times that CPU program as the step itself; that arm loads nothing of the product (its sample comes from
the numpy twin of the generator).
"""
import argparse
import ctypes
import json
import os
import resource
import shutil
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
DATA = os.path.join(ROOT, "tests", "golden", "data")
REFBIN = os.path.join(ROOT, "oracle", "_ref")
SEED = 0xB200


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


def measured_hbm_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(path))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (measured copy bandwidth)"
    except Exception:
        return 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md; MEASURED_PEAKS.json absent)"


class ClockSampler:
    """SM clock and throttle reasons sampled every few ms WHILE the timed region runs: NVML in a thread
    (nvidia_ml_py), nvidia-smi -lms as the fallback."""
    REASONS = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20), ("sw_power_cap", 0x4))
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
              "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = self.path = self.thread = None
        self.samples, self.reasons, self.sm_max = [], set(), None
        self.stop_flag = threading.Event()

    def _nvml_handle(self):
        import pynvml
        pynvml.nvmlInit()
        try:
            import torch
            uuid = str(torch.cuda.get_device_properties(self.gpu).uuid)
            return pynvml, pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid) if not uuid.startswith("GPU-") else uuid)
        except Exception:
            visible = os.environ.get("CUDA_VISIBLE_DEVICES", "")
            ids = [v for v in visible.split(",") if v.strip().isdigit()]
            return pynvml, pynvml.nvmlDeviceGetHandleByIndex(int(ids[self.gpu]) if self.gpu < len(ids) else self.gpu)

    def _loop(self, pynvml, h):
        while not self.stop_flag.is_set():
            try:
                self.samples.append(float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)))
                bits = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for name, bit in self.REASONS:
                    if bits & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.002)

    def start(self):
        try:
            pynvml, h = self._nvml_handle()
            self.sm_max = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            self.thread = threading.Thread(target=self._loop, args=(pynvml, h), daemon=True)
            self.thread.start()
            return
        except Exception:
            self.thread = None
        if shutil.which("nvidia-smi") is None:
            return
        fd, self.path = tempfile.mkstemp(suffix=".csv")
        os.close(fd)
        self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.FIELDS,
                                      "--format=csv,noheader,nounits", "-lms", "20"],
                                     stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0, "how": None}
        if self.thread is not None:
            self.stop_flag.set()
            self.thread.join(timeout=2)
            if self.samples:
                out.update(sm_mhz=float(np.median(self.samples)), sm_max_mhz=self.sm_max, reasons=sorted(self.reasons),
                           samples=len(self.samples), how="NVML in a thread during the timed steps")
            return out
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, reasons, smax = [], set(), None
        for line in open(self.path):
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax = float(f[2])
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        os.unlink(self.path)
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=smax, reasons=sorted(reasons), samples=len(sm),
                       how="nvidia-smi -lms 20 during the timed steps")
        return out


def kernel_fingerprint():
    """sha1 of the sources the dominant kernel is built from: a committed ncu capture describes THIS kernel only."""
    import hashlib
    h = hashlib.sha1()
    for rel in ("csrc/cuda/union_kernel.cu", "csrc/cuda/kmpb_device.cuh", "csrc/host/automaton.c"):
        try:
            h.update(open(os.path.join(ROOT, "multithreading_string_matching_b200", rel), "rb").read())
        except OSError:
            h.update(b"?")
    return h.hexdigest()


def measured_traffic(packets, payload_len):
    """DRAM bytes per launch of the dominant kernel from the committed `ncu --set full` capture of this workload
    (profiles/r02_traffic.json), or None when the workload differs or the kernel sources have changed since the capture
    (the file records their fingerprint)."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json")))
        if (int(t["packets"]) == int(packets) and int(t["payload_len"]) == int(payload_len)
                and t.get("kernel_fingerprint") == kernel_fingerprint()):
            return int(t["dram_bytes_read"]) + int(t["dram_bytes_write"])
    except Exception:
        pass
    return None


# ---- the synthetic stream without the product library -----------------------------------------------
# numpy twin of csrc/cuda/synth.cu (tests/test_host.py checks that both produce the same bytes): the reference arm
# and the CPU baselines generate their sample with it, so that no product code runs on that side.

def load_patterns_py(path):
    """serial.c:54-87: the whitespace-separated tokens of a strings file (fscanf("%s")), in order."""
    return open(path, "rb").read().split()


def _mix64(x):
    x = x + np.uint64(0x9e3779b97f4a7c15)
    x = (x ^ (x >> np.uint64(30))) * np.uint64(0xbf58476d1ce4e5b9)
    x = (x ^ (x >> np.uint64(27))) * np.uint64(0x94d049bb133111eb)
    return x ^ (x >> np.uint64(31))


def synth_stream(seed, first, count, L, plants, patterns):
    """payload bytes of packets [first, first+count) of the fixed-size stream, L bytes each -> (uint8[count*L], offsets)"""
    with np.errstate(over="ignore"):
        seed = np.uint64(seed)
        p = np.arange(count, dtype=np.uint64) + np.uint64(first)
        words = (L + 7) // 8
        j = np.arange(words, dtype=np.uint64)
        h = _mix64(seed ^ _mix64(p[:, None] * np.uint64(0x632be59bd9b4e019) + j[None, :]))
        b = h.view(np.uint8).reshape(count, words * 8).astype(np.uint32)
        out = (np.uint32(0x20) + ((b * np.uint32(95)) >> np.uint32(8))).astype(np.uint8)[:, :L].copy()
        n = len(patterns)
        for t in range(plants if n else 0):
            hp = _mix64(seed ^ _mix64(p * np.uint64(2) + np.uint64(1)) ^ np.uint64(0x504c414e54 + t))
            which = (hp % np.uint64(n)).astype(np.int64)
            lens = np.array([len(x) for x in patterns], dtype=np.int64)[which]
            ok = L >= lens + 1
            at = ((hp >> np.uint64(32)) % np.maximum(L - lens, 1).astype(np.uint64)).astype(np.int64)
            for w in np.unique(which):
                sel = np.nonzero((which == w) & ok)[0]
                pat = np.frombuffer(bytes(patterns[w]), dtype=np.uint8)
                out[sel[:, None], at[sel][:, None] + np.arange(len(pat))[None, :]] = pat[None, :]
        if L:
            out[:, L - 1] = 0
    return out.reshape(-1), np.arange(count + 1, dtype=np.uint64) * np.uint64(L)


# ---- CPU reference arm ---------------------------------------------------------------------------

def write_pcap(path, data, offsets):
    """Classic LE pcap v2.4, linktype 1, caplen == len; frame = Ethernet(0x0800) + IPv4(0x45, proto 17)
    + UDP + payload (SURVEY.md 8d)."""
    n = len(offsets) - 1
    lens = np.diff(offsets.astype(np.int64))
    with open(path, "wb") as f:
        f.write(np.array([0xA1B2C3D4, 0x00040002, 0, 0, 262144, 1], dtype="<u4").tobytes())
        if n and (lens == lens[0]).all():
            L = int(lens[0])
            rec = np.zeros((n, 16 + 42 + L), dtype=np.uint8)
            hdr = np.zeros(58, dtype=np.uint8)
            hdr[8:12] = np.frombuffer(np.uint32(42 + L).tobytes(), dtype=np.uint8)
            hdr[12:16] = hdr[8:12]
            hdr[16 + 12:16 + 14] = (0x08, 0x00)
            hdr[16 + 14] = 0x45
            hdr[16 + 16:16 + 18] = ((28 + L) >> 8, (28 + L) & 255)
            hdr[16 + 22], hdr[16 + 23] = 64, 17
            hdr[16 + 38:16 + 40] = ((8 + L) >> 8, (8 + L) & 255)
            rec[:, :58] = hdr
            rec[:, 58:] = data[: n * L].reshape(n, L)
            rec.tofile(f)
        else:
            for k in range(n):
                L = int(lens[k])
                hdr = bytearray(58)
                hdr[8:12] = hdr[12:16] = int(42 + L).to_bytes(4, "little")
                hdr[28:30] = b"\x08\x00"
                hdr[30] = 0x45
                hdr[32:34] = int(28 + L).to_bytes(2, "big")
                hdr[38], hdr[39] = 64, 17
                hdr[54:56] = int(8 + L).to_bytes(2, "big")
                f.write(hdr)
                f.write(data[int(offsets[k]):int(offsets[k + 1])].tobytes())


def run_reference_program(pcap, strings, threads, program="openmp_data"):
    """oracle/_ref/openmp_data or oracle/_ref/serial (the unmodified reference, -O2) -> (self-reported seconds,
    wall seconds, stdout).  serial.c takes no thread count and times reading the savefile too (serial.c:110-160)."""
    exe = os.path.join(REFBIN, program)

    def unlimited_stack():  # openmp_data.c:123 puts one pointer per packet on the stack
        try:
            resource.setrlimit(resource.RLIMIT_STACK, (resource.RLIM_INFINITY, resource.RLIM_INFINITY))
        except Exception:
            pass

    env = {k: v for k, v in os.environ.items() if not k.startswith("MALLOC_")}
    t0 = time.perf_counter()
    argv = [exe, pcap, strings] + ([str(threads)] if program.startswith("openmp_data") else [])
    out = subprocess.run(argv, capture_output=True, env=env, preexec_fn=unlimited_stack, check=True).stdout
    wall = time.perf_counter() - t0
    lines = out.decode("latin-1").splitlines()
    return float(lines[-1].split("=")[1].split()[0]), wall, "\n".join(lines[:-1]) + "\n"


class CpuReference:
    """The CPU arm: reference binary if it was built (kind 'reference'), else the oracle port.  Nothing of the product
    runs here: the sample comes from the numpy generator above."""

    def __init__(self, patterns, payload_len):
        self.patterns, self.payload_len = patterns, payload_len
        self.cores = os.cpu_count() or 1
        self.kind = "reference" if os.path.isfile(os.path.join(REFBIN, "openmp_data")) else "port"
        self.tmp = tempfile.mkdtemp(prefix="kmpb_ref_")

    def prepare(self, n_packets):
        self.n = n_packets
        self.data, self.offsets = synth_stream(SEED, 0, n_packets, self.payload_len, 2, self.patterns)
        if self.kind == "reference":
            self.pcap = os.path.join(self.tmp, "sample.pcap")
            write_pcap(self.pcap, self.data, self.offsets)

    def run(self, program="openmp_data"):
        """-> (seconds of the path, counts as reported)."""
        if self.kind == "reference":
            secs, wall, text = run_reference_program(self.pcap, os.path.join(DATA, "strings.txt"), self.cores, program=program)
            return secs, text
        from oracle import oracle_py
        t0 = time.perf_counter()
        counts = oracle_py.count_csr(self.data, self.offsets, self.patterns, threads=self.cores)
        return time.perf_counter() - t0, oracle_py.format_report(self.patterns, counts).decode("latin-1")

    def calibrate(self, target_seconds=12.0):
        """Pick a sample size that takes about target_seconds on this box's cores."""
        self.prepare(4000)
        secs, _ = self.run()
        rate = 4000 / max(secs, 1e-3)
        n = int(min(max(rate * target_seconds, 4000), 400_000))
        self.prepare(n)
        return n

    def sample_text(self):
        return "first %d packets x %d B of the bench stream (seed 0x%X), %s" % (
            self.n, self.payload_len, SEED,
            "oracle/_ref/openmp_data -O2 self-reported Elapsed time" if self.kind == "reference" else "oracle port (OpenMP)")

    def close(self):
        shutil.rmtree(self.tmp, ignore_errors=True)


def reference_arm(args, patterns):
    rank = env_int("RANK", 0)
    if rank != 0:
        return
    ref = CpuReference(patterns, args.payload_len)
    # each step a bounded sample, sized so that the whole --steps K --warmup W run ends within about two minutes
    n = args.ref_packets or ref.calibrate(max(1.0, min(8.0, 120.0 / max(args.warmup + args.steps, 1))))
    if args.ref_packets:
        ref.prepare(n)
    times = []
    for i in range(args.warmup + args.steps):
        secs, _ = ref.run()
        if i >= args.warmup:
            times.append(secs)
    ref.close()
    payload = n * args.payload_len
    ms = 1e3 * sum(times) / len(times)
    value = payload / (ms / 1e3) / 1e9
    line = {
        "impl": "reference", "metric": "payload_GBps", "value": value, "unit": "GB/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": "synthetic UDP pcap, %d packets x %d B payloads per GPU, bundled strings.txt (97 patterns, 87 distinct)"
                               % (args.packets, args.payload_len),
                   "sample": "each step = the first %d packets of that stream on the host cores" % n,
                   "packets_per_step": n, "payload_bytes_per_step": payload},
        "packets_per_s": n / (ms / 1e3),
        "cpu_baseline": {"value": value, "unit": "GB/s", "cores": ref.cores, "kind": ref.kind, "sample": ref.sample_text()},
        "e2e": {"value": value, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ---- our arm --------------------------------------------------------------------------------------

class Dist:
    """rank / world plumbing shared by the configurations"""

    def __init__(self):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.rank, self.world, self.local = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
        if self.world > 1:
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, x):
        if self.world == 1:
            return x
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(self, x):
        if self.world == 1:
            return x
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t)
        return float(t.item())

    def close(self):
        if self.world > 1:
            self.dist.destroy_process_group()


def symmetric_rows(D, rows, n_pat):
    """rows x n_pat int64 count vectors in symmetric memory (mapped into all ranks over NVLink), or None"""
    torch, dist = D.torch, D.dist
    ok, why, sym, ptrs = 1, "", None, None
    try:
        import torch.distributed._symmetric_memory as symm
        sym = symm.empty((rows, n_pat), dtype=torch.int64, device=D.dev)
        sym.zero_()
        hdl = symm.rendezvous(sym, dist.group.WORLD)
        ptrs = [int(hdl.buffer_ptrs[r]) for r in range(D.world)]
    except Exception as e:  # no symmetric memory on this box / build
        ok, why = 0, repr(e)[:200]
    agree = torch.tensor([ok], dtype=torch.int32, device=D.dev)
    dist.all_reduce(agree, op=dist.ReduceOp.MIN)
    torch.cuda.synchronize()
    dist.barrier()
    if int(agree.item()) == 1:
        return {"sym": sym, "ptrs": ptrs, "rows": rows}
    if D.rank == 0 and why:
        print("bench: symmetric memory unavailable, using NCCL all-reduce: " + why, file=sys.stderr)
    return None


def timed_passes(D, fn, steps, warmup=3):
    """ms per call of fn(), CUDA events on the current stream, barrier on both sides, max over ranks"""
    torch = D.torch
    for _ in range(warmup):
        fn()
    D.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    D.barrier()
    return D.max_over_ranks(e0.elapsed_time(e1)) / steps


def h2d_peak(D, nbytes, reps=3):
    """What bare pinned cudaMemcpyAsync copies reach when every rank copies at once (GB/s summed over ranks): the
    ceiling of the end-to-end number, measured in the same run (the Scatterv of mpi_dumping.c:161 done by copy engines)."""
    torch = D.torch
    nbytes = int(min(nbytes, 2 << 30))
    h = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
    d = torch.empty(nbytes, dtype=torch.uint8, device=D.dev)
    d.copy_(h, non_blocking=True)
    D.barrier()
    t0 = time.perf_counter()
    for _ in range(reps):
        d.copy_(h, non_blocking=True)
    D.barrier()
    dt = D.max_over_ranks(time.perf_counter() - t0)
    del h, d
    return D.sum_over_ranks(float(nbytes)) * reps / dt / 1e9


def dump_outputs(out_dir, **arrays):
    """DIR/<name>.npy for each array, as float64: exact for integer counts below 2**53, so that the outputs of two
    builds on the same seeded stream can be compared value for value."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float64))


def oracle_prefix_ok(kmp, m, patterns, data, offsets, n):
    """counts of the first n packets through the C ABI's host form == the oracle's (bit-exact)"""
    from oracle import oracle_py
    n = min(n, len(offsets) - 1)
    sub_off = np.ascontiguousarray(offsets[: n + 1]).astype(np.uint64)
    sub = np.ascontiguousarray(data[: int(sub_off[-1])])
    return m.count_host(sub, sub_off) == oracle_py.count_csr(sub, sub_off, patterns)


def ours(args, kmp, patterns):
    D = Dist()
    torch, dist, dev, rank, world, local = D.torch, D.dist, D.dev, D.rank, D.world, D.local

    per_gpu = args.packets
    total_packets = per_gpu * world                      # weak scaling: the stream grows with N
    from multithreading_string_matching_b200 import distributed as kd
    first, count = kd.rank_slice(total_packets, rank, world)   # mpi_dumping.c:149-157
    L = args.payload_len
    n_pat = len(patterns)
    m = kmp.Matcher(local, engine=args.engine)
    m.set_patterns(patterns)
    synth = kmp.Synth(seed=SEED, payload_len=L, plants=2, plant_patterns=patterns)
    nbytes = synth.nbytes(first, count)
    d_bytes = torch.empty(nbytes + 4096, dtype=torch.uint8, device=dev)
    d_bytes[nbytes:].zero_()
    d_off = torch.empty(count + 1, dtype=torch.int64, device=dev)
    synth.fill_device(m, first, count, d_bytes.data_ptr(), d_off.data_ptr())
    # two count vectors: the all-reduce of step i runs on a side stream while step i+1's kernel matches the
    # next batch (in a pipeline the batches differ; here it is the same slice again)
    d_counts2 = [torch.zeros(n_pat, dtype=torch.int64, device=dev) for _ in range(2)]
    d_counts = d_counts2[0]
    torch.cuda.synchronize()
    stream = torch.cuda.current_stream()
    side = torch.cuda.Stream(device=dev) if world > 1 else None
    reduced = [None, None]
    step_no = [0]

    # Reduce across GPUs.  Preferred: every rank's count vectors live in symmetric memory (mapped into all
    # ranks over NVLink) and the match kernel's last block adds its counts straight into all of them --
    # no collective call at all (kmpb_count_device_span_peers).  One row of counts per step, so no rank
    # ever clears a vector another rank may be adding to.  Fallback: one NCCL all-reduce per step on a
    # side stream, overlapped with the next step's kernel.
    p2p = None
    if world > 1 and args.reduce != "nccl" and args.engine == "union":
        p2p = symmetric_rows(D, 2 * (args.warmup + args.steps) + 64, n_pat)

    def step():
        if p2p is not None:
            row = step_no[0] % p2p["rows"]
            step_no[0] += 1
            vecs = [ptr + row * n_pat * 8 for ptr in p2p["ptrs"]]
            m.count_device_into(d_bytes.data_ptr(), d_off.data_ptr(), count, vecs, span=(0, nbytes), stream=stream.cuda_stream)
            return p2p["sym"][row]
        i = step_no[0] & 1
        step_no[0] += 1
        buf = d_counts2[i]
        if reduced[i] is not None:
            stream.wait_event(reduced[i])  # the vector's previous all-reduce has read it
        buf.zero_()
        m.count_device(d_bytes.data_ptr(), d_off.data_ptr(), count, buf.data_ptr(), span=(0, nbytes),
                       stream=stream.cuda_stream)
        if world > 1:
            ready = torch.cuda.Event()
            ready.record(stream)
            with torch.cuda.stream(side):
                side.wait_event(ready)
                kd.reduce_counts(buf)  # the MPI_Reduce(SUM) of mpi_dumping.c:202, as an NCCL all-reduce over NVLink
                reduced[i] = torch.cuda.Event()
                reduced[i].record(side)
        return buf

    def drain_side():
        if world > 1 and p2p is None:
            stream.wait_stream(side)

    barrier, max_over_ranks = D.barrier, D.max_over_ranks

    # ---- device-resident timing -------------------------------------------------------------------
    for _ in range(args.warmup):
        step()
    drain_side()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = m.launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        d_counts = step()
    drain_side()  # the last all-reduce is inside the timed region
    e1.record()
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    ms_step = max_over_ranks(e0.elapsed_time(e1)) / args.steps
    launches = m.launches - launches0  # partition + union + count expansion per step (libkmpb200's own counter)
    counts_resident = d_counts.cpu().numpy().copy()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, counts=counts_resident)

    # ---- the dominant kernel alone (roofline) -----------------------------------------------------
    m.set_profile(True)
    kms = []
    for _ in range(max(3, min(args.steps, 10))):
        step()
        kms.append(m.last_kernel_ms())
    drain_side()
    m.set_profile(False)
    barrier()
    kernel_ms = max_over_ranks(float(np.mean(kms)))
    algo_bytes = nbytes + 8 * (count + 1)  # payload once + one offset per packet (DESIGN.md section 5)
    peak, peak_src = measured_hbm_peak()
    achieved = algo_bytes / (kernel_ms / 1e3) / 1e9

    # ---- this rank's own counts, and parity at full size: the per-pattern engine over the whole slice ----------
    # (the prescribed one-DFA-per-pattern design, an independent implementation on the device; ~0.3 s for 14 GB)
    d_own = torch.zeros(n_pat, dtype=torch.int64, device=dev)
    m.count_device(d_bytes.data_ptr(), d_off.data_ptr(), count, d_own.data_ptr(), span=(0, nbytes), stream=stream.cuda_stream)
    torch.cuda.synchronize()
    own_counts = d_own.cpu().numpy().copy()
    parity_full = None
    if args.engine == "union" and not args.no_parity:
        m.set_engine("perpat")
        d_pp = torch.zeros(n_pat, dtype=torch.int64, device=dev)
        m.count_device(d_bytes.data_ptr(), d_off.data_ptr(), count, d_pp.data_ptr(), span=(0, nbytes), stream=stream.cuda_stream)
        torch.cuda.synchronize()
        m.set_engine("union")
        parity_full = bool(np.array_equal(d_pp.cpu().numpy(), own_counts))
        if world > 1:
            t = torch.tensor([1 if parity_full else 0], dtype=torch.int32, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
            parity_full = bool(int(t.item()))
        del d_pp
    if world == 1:
        assert np.array_equal(own_counts, counts_resident), "two passes over the same slice disagree"

    # ---- strong scaling: the FIXED stream of one GPU's size split over the ranks (mpi_dumping.c:149-157) --------
    strong = None
    if world > 1 and args.engine == "union":
        sfirst, scount = kd.rank_slice(per_gpu, rank, world)
        sbytes = synth.nbytes(sfirst, scount)
        s_bytes = torch.empty(sbytes + 4096, dtype=torch.uint8, device=dev)
        s_bytes[sbytes:].zero_()
        s_off = torch.empty(scount + 1, dtype=torch.int64, device=dev)
        synth.fill_device(m, sfirst, scount, s_bytes.data_ptr(), s_off.data_ptr())
        torch.cuda.synchronize()
        srow = [0]
        s_local = torch.zeros(n_pat, dtype=torch.int64, device=dev)

        def strong_step():
            if p2p is not None:
                row = (step_no[0] + srow[0]) % p2p["rows"]
                srow[0] += 1
                vecs = [ptr + row * n_pat * 8 for ptr in p2p["ptrs"]]
                m.count_device_into(s_bytes.data_ptr(), s_off.data_ptr(), scount, vecs, span=(0, sbytes), stream=stream.cuda_stream)
            else:
                s_local.zero_()
                m.count_device(s_bytes.data_ptr(), s_off.data_ptr(), scount, s_local.data_ptr(), span=(0, sbytes), stream=stream.cuda_stream)
                kd.reduce_counts(s_local)

        ssteps = max(3, min(args.steps, 20))
        ms_strong = timed_passes(D, strong_step, ssteps)
        # the summed counts must be those of the whole stream = rank 0's own slice of the weak run (packets 0 .. per_gpu)
        s_local.zero_()
        m.count_device(s_bytes.data_ptr(), s_off.data_ptr(), scount, s_local.data_ptr(), span=(0, sbytes), stream=stream.cuda_stream)
        kd.reduce_counts(s_local)
        whole = torch.as_tensor(own_counts, device=dev).clone()
        dist.broadcast(whole, src=0)
        strong_ok = bool(torch.equal(whole, s_local))
        strong = {"packets_total": per_gpu, "payload_bytes_total": per_gpu * L, "ms_per_step": ms_strong,
                  "value": per_gpu * L / (ms_strong / 1e3) / 1e9, "unit": "GB/s",
                  "ms_per_step_one_gpu_same_run": ms_step, "efficiency_vs_n1": (ms_step / world) / ms_strong,
                  "steps": ssteps, "counts_match_unsplit_stream": strong_ok,
                  "what": "the %d-packet stream of ONE GPU split over %d ranks (N/P packets each, rank 0 also N%%P), "
                          "reduce as in the weak run; one-GPU time = this run's per-rank pass over a slice of that size" % (per_gpu, world)}
        del s_bytes, s_off

    # ---- end to end through the host entry point -------------------------------------------------
    e2e = None
    if not args.no_e2e:
        import psutil
        need = (nbytes + 8 * (count + 1)) * world
        e2e_count = count
        if psutil.virtual_memory().available < 2.5 * need:
            e2e_count = max(int(count * psutil.virtual_memory().available / (3.0 * need)), 1000)
        e_bytes = synth.nbytes(first, e2e_count)
        peak_h2d = h2d_peak(D, e_bytes)
        h_bytes = torch.empty(e_bytes + 4096, dtype=torch.uint8, pin_memory=True)
        h_off = torch.empty(e2e_count + 1, dtype=torch.int64, pin_memory=True)
        h_bytes[: e_bytes].copy_(d_bytes[: e_bytes])
        h_off.copy_(d_off[: e2e_count + 1])
        torch.cuda.synchronize()
        e2e_steps = max(1, min(args.steps, 5))

        def e2e_step():
            c = m.count_host_ptr(h_bytes.data_ptr(), h_off.data_ptr(), e2e_count)
            if world > 1:
                t = torch.tensor(c, dtype=torch.int64, device=dev)
                dist.all_reduce(t)
                c = t.cpu().tolist()
            return c

        c = e2e_step()
        barrier()
        t0 = time.perf_counter()
        e0.record()
        for _ in range(e2e_steps):
            c = e2e_step()
        e1.record()
        barrier()
        wall_ms = 1e3 * (time.perf_counter() - t0) / e2e_steps
        e2e_ms = max_over_ranks(max(e0.elapsed_time(e1) / e2e_steps, wall_ms))
        if e2e_count == count:
            assert np.array_equal(np.asarray(c, dtype=np.int64), counts_resident), "host and device paths disagree"
        e2e_total = D.sum_over_ranks(float(e_bytes))
        e2e_val = e2e_total / (e2e_ms / 1e3) / 1e9
        e2e = {"value": e2e_val, "unit": "GB/s", "ms_per_step": e2e_ms,
               "h2d_bytes_per_step": int(e_bytes + 8 * (e2e_count + 1)), "d2h_bytes_per_step": int(8 * n_pat),
               "packets_per_step_per_gpu": int(e2e_count), "steps": e2e_steps,
               "h2d_peak_gbs": peak_h2d, "frac_of_h2d_peak": e2e_val / peak_h2d,
               "h2d_peak_how": "bare pinned cudaMemcpyAsync of the same size on every rank at once, this run (host link ceiling)",
               "note": "kmpb_count_host: pinned host CSR -> 64 MiB chunks over 4 streams (H2D overlapped with kernels) -> counts D2H"
                       + ("" if e2e_count == count else "; REDUCED sample: host RAM too small for the full slice")}
        del h_bytes, h_off

    total_bytes = D.sum_over_ranks(float(nbytes))

    # ---- the other configurations, small forms (the full ones: --config c4 | c5) ---------------------------------
    sweep = None
    if not args.no_sweep and args.engine == "union":
        d_bytes = d_off = None
        torch.cuda.empty_cache()
        sweep = {"c4": config_c4(D, kmp, m, cells=[(1, 8), (16, 16), (64, 32), (256, 64)], payload_bytes=250_000_000, steps=3),
                 "c5": config_c5(D, kmp, m, patterns, total_packets=1_368_000, steps=5, e2e=False)}
        m.set_engine("union")
        m.set_patterns(patterns)
        d_bytes = torch.empty(nbytes + 4096, dtype=torch.uint8, device=dev)
        d_bytes[nbytes:].zero_()
        d_off = torch.empty(count + 1, dtype=torch.int64, device=dev)
        synth.fill_device(m, first, count, d_bytes.data_ptr(), d_off.data_ptr())

    if rank == 0:
        value = total_bytes / (ms_step / 1e3) / 1e9
        line = {
            "metric": "payload_GBps", "value": value, "unit": "GB/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": "synthetic UDP pcap, %d packets x %d B payloads per GPU, bundled strings.txt (97 patterns, 87 distinct)"
                                   % (per_gpu, L),
                       "packets_total": total_packets, "payload_bytes_total": int(total_bytes), "engine": args.engine,
                       "split": "mpi_dumping.c:149-157 contiguous packet slices",
                       "reduce": ("none (one GPU)" if world == 1 else
                                  "in the match kernel: its last block adds the counts to every rank's vector in symmetric memory over NVLink (no collective call)"
                                  if p2p is not None else "one NCCL all-reduce per step on a side stream, overlapped with the next step's kernel"),
                       "l2": "inputs (%.1f GB per GPU) larger than the 126 MB L2; no flush needed" % (nbytes / 1e9)},
            "packets_per_s": total_packets / (ms_step / 1e3),
            "hbm_frac_of_measured_peak": value / world / peak,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": measured_traffic(count, L) if args.engine != "perpat" else None, "kernel": "kmpb_union_kernel" if args.engine != "perpat" else "kmpb_perpat_kernel",
                         "kernel_ms": kernel_ms, "algorithmic_bytes_per_launch": int(algo_bytes), "peak_source": peak_src,
                         "kernel_fingerprint": kernel_fingerprint()},
            "e2e": e2e, "gpu_launches": int(launches), "gpu_launches_per_step": int(launches) // max(args.steps, 1), "clocks": clocks,
            "matches_per_step": int(counts_resident.sum()),
            "parity_full": parity_full,
            "parity_full_how": "kmpb_perpat_kernel (one KMP DFA per pattern, the reference's loop as written) over every rank's whole slice == the union engine's counts",
        }
        if strong is not None:
            line["strong"] = strong
        if sweep is not None:
            line["sweep"] = sweep
        if world == 1 and not args.no_cpu:
            ref = CpuReference(patterns, L)
            n = args.ref_packets or ref.calibrate(12.0)
            if args.ref_packets:
                ref.prepare(n)
            secs, text = ref.run()

            def ours_on_prefix(k):  # parity at bench time: our counts on the same prefix must print the same lines
                d_c = torch.zeros(n_pat, dtype=torch.int64, device=dev)
                m.count_device(d_bytes.data_ptr(), d_off.data_ptr(), k, d_c.data_ptr(), span=(0, k * L), stream=stream.cuda_stream)
                torch.cuda.synchronize()
                return kmp.format_report(patterns, d_c.cpu().tolist()).decode("latin-1")

            line["cpu_baseline"] = {"value": n * L / secs / 1e9, "unit": "GB/s", "cores": ref.cores, "kind": ref.kind,
                                    "sample": ref.sample_text(), "seconds": secs, "counts_match_gpu": ours_on_prefix(n) == text}
            if ref.kind == "reference":
                strings = os.path.join(DATA, "strings.txt")

                def other(program, k, cores, what):
                    if not os.path.isfile(os.path.join(REFBIN, program)):
                        return None
                    pc = os.path.join(ref.tmp, program + ".pcap")
                    write_pcap(pc, ref.data[: k * L], ref.offsets[: k + 1])
                    s, _, t = run_reference_program(pc, strings, cores, program=program)
                    os.unlink(pc)
                    return {"value": k * L / s / 1e9, "unit": "GB/s", "cores": cores, "seconds": s,
                            "sample": "first %d packets of the same stream, %s" % (k, what), "counts_match_gpu": ours_on_prefix(k) == t}
                # serial.c, the one-core form of the same loop, on a prefix of that sample sized for a few seconds
                ns = max(min(n // (2 * ref.cores), n), 1000)
                line["cpu_baseline"]["serial"] = other(
                    "serial", ns, 1, "oracle/_ref/serial -O2 self-reported Elapsed time (includes reading the savefile)")
                # the documented compile lines (no -O flag): serial.c:2, openmp_data.c:1
                line["cpu_baseline"]["openmp_data_documented_flags"] = other(
                    "openmp_data_doc", max(n // 3, 1000), ref.cores, "oracle/_ref/openmp_data_doc (gcc -g -Wall -fopenmp, openmp_data.c:1)")
                line["cpu_baseline"]["serial_documented_flags"] = other(
                    "serial_doc", max(ns // 2, 500), 1, "oracle/_ref/serial_doc (gcc -g, serial.c:2)")
                # the step before the path (SURVEY 8f): savefile -> pinned CSR batch, on the same sample pcap
                t0 = time.perf_counter()
                batch = kmp.PayloadBatch(ref.pcap, "udp", pinned=True)
                dt = time.perf_counter() - t0
                line["ingest"] = {"value": batch.total_bytes / dt / 1e9, "unit": "GB/s", "seconds": dt, "packets": int(batch.n_packets),
                                  "what": "kmpb_load_pcap_csr (mmap, record framing, OpenMP pack into pinned memory) on the CPU sample's pcap"}
                batch.close()
            ref.close()
        print(json.dumps(line), flush=True)
    m.close()
    D.close()


# ---- BASELINE configs[3]: pattern sweep (DFA shared-memory pressure) ------------------------------------------------

def sweep_patterns(n, length, seed=0xC4):
    """n distinct random [a-z0-9] patterns of `length` bytes from the stream's PRNG"""
    alpha = np.frombuffer(b"abcdefghijklmnopqrstuvwxyz0123456789", dtype=np.uint8)
    out, seen, k = [], set(), 0
    with np.errstate(over="ignore"):
        while len(out) < n:
            h = _mix64(np.uint64(seed) ^ _mix64(np.arange(k, k + length, dtype=np.uint64) + np.uint64((n * 131 + length) << 20)))
            p = bytes(alpha[(h % np.uint64(36)).astype(np.int64)])
            k += length
            if p not in seen:
                seen.add(p)
                out.append(p)
    return out


def config_c4(D, kmp, m, cells=None, payload_bytes=1_000_000_000, steps=5, L=1400):
    """1..256 patterns of 4..64 bytes over `payload_bytes` of synthetic payload (two of the set's patterns planted per
    packet, so there are matches): the union engine and the per-pattern engine (whose DFAs are tiled through shared memory
    when they exceed it) on the same bytes, counts cross-checked between them and, on a prefix, against the oracle."""
    torch = D.torch
    if cells is None:
        cells = [(n, ln) for n in (1, 2, 4, 8, 16, 32, 64, 128, 256) for ln in (4, 8, 16, 32, 64)]
    count = payload_bytes // L
    stream = torch.cuda.current_stream()
    d_bytes = torch.empty(count * L + 4096, dtype=torch.uint8, device=D.dev)
    d_bytes[count * L:].zero_()
    d_off = torch.empty(count + 1, dtype=torch.int64, device=D.dev)
    rows = []
    for n, ln in cells:
        pats = sweep_patterns(n, ln)
        synth = kmp.Synth(seed=SEED + 4, payload_len=L, plants=2, plant_patterns=pats)
        m.set_engine("union")
        m.set_patterns(pats)
        synth.fill_device(m, 0, count, d_bytes.data_ptr(), d_off.data_ptr())
        d_c = torch.zeros(n, dtype=torch.int64, device=D.dev)
        res = {}
        for engine in ("union", "perpat"):
            m.set_engine(engine)
            m.set_profile(True)
            ms = []
            for i in range(steps if engine == "union" else max(1, steps // 2)):
                d_c.zero_()
                m.count_device(d_bytes.data_ptr(), d_off.data_ptr(), count, d_c.data_ptr(), span=(0, count * L), stream=stream.cuda_stream)
                ms.append(m.last_kernel_ms())
            m.set_profile(False)
            res[engine] = (float(np.mean(ms[1:] or ms)), d_c.cpu().numpy().copy())
        m.set_engine("union")
        hd, ho = synth.fill_host(0, 300)
        rows.append({"patterns": n, "length": ln,
                     "union_GBps": count * L / res["union"][0] / 1e6, "perpat_GBps": count * L / res["perpat"][0] / 1e6,
                     "matches": int(res["union"][1].sum()), "engines_agree": bool(np.array_equal(res["union"][1], res["perpat"][1])),
                     "oracle_prefix_ok": bool(oracle_prefix_ok(kmp, m, pats, hd, ho, 300)),
                     "perpat_dfa_bytes": n * ln * 256})
    del d_bytes, d_off
    torch.cuda.empty_cache()
    peak, _ = measured_hbm_peak()
    return {"payload_bytes": count * L, "text": "printable synthetic payloads, 2 patterns of the cell's set planted per packet, last byte NUL",
            "unit": "GB/s (kernel alone, CUDA events on its stream)", "hbm_peak": peak, "cells": rows,
            "all_agree": all(r["engines_agree"] and r["oracle_prefix_ok"] for r in rows)}


# ---- BASELINE configs[4]: mixed 64..9000-byte payloads, end to end, over the ranks ------------------------------------

def config_c5(D, kmp, m, patterns, total_packets=6_840_000, steps=10, e2e=True):
    """Packet lengths drawn from {64: 40 %, 576: 20 %, 1400: 30 %, 9000: 10 %} (seeded), ~10 GB in all, split over the
    ranks as mpi_dumping.c:149-157 splits packets; device-resident with the reduce inside the match kernel (NCCL when
    there is no symmetric memory), and end to end from pinned host memory through kmpb_count_host + all-reduce."""
    torch, dist = D.torch, D.dist
    from multithreading_string_matching_b200 import distributed as kd
    n_pat = len(patterns)
    m.set_engine("union")
    m.set_patterns(patterns)
    synth = kmp.Synth(seed=11, len_mode=1, plants=2, plant_patterns=patterns)
    first, count = kd.rank_slice(total_packets, D.rank, D.world)
    nbytes = synth.nbytes(first, count)
    d_bytes = torch.empty(nbytes + 4096, dtype=torch.uint8, device=D.dev)
    d_bytes[nbytes:].zero_()
    d_off = torch.empty(count + 1, dtype=torch.int64, device=D.dev)
    synth.fill_device(m, first, count, d_bytes.data_ptr(), d_off.data_ptr())
    torch.cuda.synchronize()
    stream = torch.cuda.current_stream()
    p2p = symmetric_rows(D, steps + 16, n_pat) if D.world > 1 else None
    d_c = torch.zeros(n_pat, dtype=torch.int64, device=D.dev)
    it = [0]

    def device_step():
        if p2p is not None:
            row = it[0] % p2p["rows"]
            it[0] += 1
            vecs = [ptr + row * n_pat * 8 for ptr in p2p["ptrs"]]
            m.count_device_into(d_bytes.data_ptr(), d_off.data_ptr(), count, vecs, span=(0, nbytes), stream=stream.cuda_stream)
        else:
            d_c.zero_()
            m.count_device(d_bytes.data_ptr(), d_off.data_ptr(), count, d_c.data_ptr(), span=(0, nbytes), stream=stream.cuda_stream)
            kd.reduce_counts(d_c)

    ms_dev = timed_passes(D, device_step, steps)
    total_bytes = D.sum_over_ranks(float(nbytes))
    # parity: both engines on this rank's slice, the oracle on a prefix of it
    own = torch.zeros(n_pat, dtype=torch.int64, device=D.dev)
    m.count_device(d_bytes.data_ptr(), d_off.data_ptr(), count, own.data_ptr(), span=(0, nbytes), stream=stream.cuda_stream)
    m.set_engine("perpat")
    pp = torch.zeros(n_pat, dtype=torch.int64, device=D.dev)
    m.count_device(d_bytes.data_ptr(), d_off.data_ptr(), count, pp.data_ptr(), span=(0, nbytes), stream=stream.cuda_stream)
    torch.cuda.synchronize()
    m.set_engine("union")
    hd, ho = synth.fill_host(first, 2000)
    ok = bool(torch.equal(own, pp)) and bool(oracle_prefix_ok(kmp, m, patterns, hd, ho, 2000))
    ok = bool(D.max_over_ranks(0.0 if ok else 1.0) == 0.0)
    total = own.clone()
    kd.reduce_counts(total)
    out = {"packets_total": total_packets, "payload_bytes_total": int(total_bytes), "n_gpus": D.world,
           "device_GBps": total_bytes / (ms_dev / 1e3) / 1e9, "device_ms_per_step": ms_dev, "steps": steps,
           "reduce": "none (one GPU)" if D.world == 1 else ("in the match kernel over symmetric memory" if p2p is not None else "NCCL all-reduce per step"),
           "parity": ok, "parity_how": "union == per-pattern engine on every rank's whole slice; first 2000 packets of every slice == oracle",
           "matches": int(total.sum().item())}
    if e2e:
        peak_h2d = h2d_peak(D, nbytes)
        h_bytes = torch.empty(nbytes + 4096, dtype=torch.uint8, pin_memory=True)
        h_off = torch.empty(count + 1, dtype=torch.int64, pin_memory=True)
        h_bytes[:nbytes].copy_(d_bytes[:nbytes])
        h_off.copy_(d_off)
        torch.cuda.synchronize()

        def host_step():
            c = m.count_host_ptr(h_bytes.data_ptr(), h_off.data_ptr(), count)
            t = torch.tensor(c, dtype=torch.int64, device=D.dev)
            kd.reduce_counts(t)
            return t

        c = host_step()
        D.barrier()
        t0 = time.perf_counter()
        for _ in range(max(1, steps // 2)):
            c = host_step()
        D.barrier()
        ms_e2e = D.max_over_ranks(1e3 * (time.perf_counter() - t0) / max(1, steps // 2))
        out.update({"e2e_GBps": total_bytes / (ms_e2e / 1e3) / 1e9, "e2e_ms_per_step": ms_e2e, "h2d_peak_gbs": peak_h2d,
                    "e2e_frac_of_h2d_peak": total_bytes / (ms_e2e / 1e3) / 1e9 / peak_h2d,
                    "e2e_counts_match_device": bool(torch.equal(c, total))})
        del h_bytes, h_off
    del d_bytes, d_off
    torch.cuda.empty_cache()
    return out


def run_config(args, kmp, patterns):
    """--config c4 | c5 | cli: one JSON line for that configuration"""
    D = Dist()
    m = kmp.Matcher(D.local, engine="union")
    if args.config == "c4":
        body = config_c4(D, kmp, m) if D.rank == 0 or D.world == 1 else None
        line = {"metric": "payload_GBps", "config": {"workload": "BASELINE configs[3]: pattern sweep, 1-256 patterns x 4-64 bytes over 1 GB"},
                "n_gpus": 1, "sweep": body}
    elif args.config == "c5":
        body = config_c5(D, kmp, m, patterns, steps=max(3, min(args.steps, 10)))
        line = {"metric": "payload_GBps", "unit": "GB/s", "n_gpus": D.world, "value": body["device_GBps"],
                "config": {"workload": "BASELINE configs[4]: mixed 64/576/1400/9000-byte payloads (40/20/30/10 % of the packets), ~10 GB, strings.txt"},
                "e2e": {"value": body.get("e2e_GBps"), "unit": "GB/s"}, "c5": body}
    else:
        body = config_cli(args, kmp, patterns) if D.rank == 0 else None
        line = {"metric": "payload_GBps", "config": {"workload": "process level: bin/kmp_match on a synthetic savefile (config 3's stream)"},
                "n_gpus": 1, "process_e2e": body}
    if D.rank == 0:
        print(json.dumps(line), flush=True)
    m.close()
    D.close()


# ---- the drop-in command line on a large savefile -----------------------------------------------------------------------

def config_cli(args, kmp, patterns):
    """bin/kmp_match <pcap> <strings> on a savefile of config 3's stream in /dev/shm: wall time of the whole process and
    the stages it reports (KMPB_STATS), next to oracle/_ref/openmp_data on a prefix of the same file (its rate does not
    depend on the file size; the whole file would take it minutes) with the outputs compared on that prefix."""
    L = args.payload_len
    tmp = tempfile.mkdtemp(prefix="kmpb_cli_", dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
    strings = os.path.join(DATA, "strings.txt")
    exe = os.path.join(ROOT, "multithreading_string_matching_b200", "bin", "kmp_match")
    out = {}
    try:
        n_big = int(args.cli_gb * 1e9 // (L + 58))
        big = os.path.join(tmp, "big.pcap")
        chunk = 200_000
        with open(big, "wb") as f:
            f.write(np.array([0xA1B2C3D4, 0x00040002, 0, 0, 262144, 1], dtype="<u4").tobytes())
        gen = kmp.Synth(seed=SEED, payload_len=L, plants=2, plant_patterns=patterns)  # same bytes as synth_stream, OpenMP
        for k0 in range(0, n_big, chunk):
            k = min(chunk, n_big - k0)
            data, offs = gen.fill_host(k0, k)
            part = os.path.join(tmp, "part.pcap")
            write_pcap(part, data, offs)
            with open(big, "ab") as f, open(part, "rb") as g:
                g.seek(24)
                shutil.copyfileobj(g, f, 1 << 24)
            os.unlink(part)
        size = os.path.getsize(big)
        runs = []
        for i in range(3):
            t0 = time.perf_counter()
            r = subprocess.run([exe, big, strings], capture_output=True, env=dict(os.environ, KMPB_STATS="1"))
            wall = time.perf_counter() - t0
            text = r.stdout.decode("latin-1")
            runs.append({"wall_s": wall, "self_reported_s": float(text.strip().splitlines()[-1].split("=")[1].split()[0]),
                         "stats": r.stderr.decode("latin-1").strip().splitlines()[-6:]})
        best = min(runs, key=lambda x: x["wall_s"])
        out.update({"savefile_bytes": size, "packets": n_big, "payload_bytes": n_big * L, "runs": runs,
                    "payload_GBps_wall": n_big * L / best["wall_s"] / 1e9,
                    "payload_GBps_self_reported": n_big * L / best["self_reported_s"] / 1e9})
        # the reference program on a prefix, outputs compared
        n_small = min(n_big, 200_000)
        small = os.path.join(tmp, "small.pcap")
        data, offs = synth_stream(SEED, 0, n_small, L, 2, patterns)
        write_pcap(small, data, offs)
        if os.path.isfile(os.path.join(REFBIN, "openmp_data")):
            secs, wall, ref_text = run_reference_program(small, strings, os.cpu_count() or 1)
            r = subprocess.run([exe, small, strings], capture_output=True)
            ours_text = "\n".join(r.stdout.decode("latin-1").splitlines()[:-1]) + "\n"
            out["reference_on_prefix"] = {"packets": n_small, "openmp_data_self_reported_s": secs, "openmp_data_wall_s": wall,
                                          "openmp_data_GBps": n_small * L / secs / 1e9, "cores": os.cpu_count(),
                                          "outputs_identical": ours_text == ref_text}
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="c3", choices=["c3", "c4", "c5", "cli"],
                    help="c3 (default): BASELINE configs[2], the headline; c4: pattern sweep; c5: mixed payload sizes; cli: bin/kmp_match on a large savefile")
    ap.add_argument("--packets", type=int, default=10_000_000, help="packets per GPU (BASELINE config 3: 10 M)")
    ap.add_argument("--payload-len", type=int, default=1400)
    ap.add_argument("--engine", default="union", choices=["union", "perpat"])
    ap.add_argument("--ref-packets", type=int, default=0, help="CPU sample size (0 = calibrate to ~10 s)")
    ap.add_argument("--reduce", default="auto", choices=["auto", "nccl"], help="N>1: in-kernel reduce over symmetric memory, or NCCL")
    ap.add_argument("--cli-gb", type=float, default=10.0, help="--config cli: size of the savefile")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-sweep", action="store_true", help="skip the small forms of configs 4 and 5 on the default line")
    ap.add_argument("--no-parity", action="store_true", help="skip the full-size cross-check against the per-pattern engine")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned (the count vector) as DIR/counts.npy, float64")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.config != "c3"):
        ap.error("--dump-outputs writes the outputs of the default configuration (--impl ours --config c3)")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    # stdout carries the one JSON line and nothing else: whatever libraries write to file descriptor 1 in the
    # meantime (NCCL prints its version there when the box sets NCCL_DEBUG) goes to stderr
    sys.stdout.flush()
    json_out = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    sys.stdout = json_out

    if args.impl == "reference":
        # the reference arm runs the unmodified reference program (or the oracle port) on a sample made by the numpy
        # generator: no product library is loaded on this side
        reference_arm(args, load_patterns_py(os.path.join(DATA, "strings.txt")))
        return

    import multithreading_string_matching_b200 as kmp  # raises if libkmpb200.so is missing: no fallback

    patterns = kmp.load_patterns(os.path.join(DATA, "strings.txt"))
    if args.config == "c3":
        ours(args, kmp, patterns)
    else:
        run_config(args, kmp, patterns)


if __name__ == "__main__":
    main()
