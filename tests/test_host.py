"""Host side of the product (C code in libkmpb200.so) against the oracle and the golden vectors.
CPU only: nothing here launches a kernel."""
import ctypes
import json
import os
import re
import struct
import subprocess

import numpy as np
import pytest

from conftest import DATA, GOLDEN, ROOT
from kmpb_harness import MATCH, PCAPS, build_integration_snippet, pcapng, udp_frame, write_pcap

import multithreading_string_matching_b200 as kmp

HOSTC = os.path.join(ROOT, "multithreading_string_matching_b200", "csrc", "host")


def test_library_exports_every_declared_symbol():
    """Every function include/kmpb200.h declares is exported by the built library and bound."""
    header = open(os.path.join(ROOT, "include", "kmpb200.h")).read()
    declared = set(re.findall(r"\b(kmpb_[a-z0-9_]+)\s*\(", header))
    declared -= {"kmpb_ctx"}
    assert len(declared) >= 25
    lib = kmp.lib()
    for name in sorted(declared):
        assert hasattr(lib, name), name
    assert declared == set(kmp.SIGNATURES), declared ^ set(kmp.SIGNATURES)
    assert lib.kmpb_version() == b"0.1.0"


def test_no_cpu_fallback_without_a_device():
    """Without a B200 the matcher refuses to exist: the product has no CPU path."""
    import torch

    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    assert kmp.device_count() == 0
    with pytest.raises(kmp.KmpbError) as e:
        kmp.Matcher()
    assert e.value.code == -4


def test_product_does_not_touch_the_oracle():
    """Nothing under the package may import, link or execute oracle/."""
    pkg = os.path.join(ROOT, "multithreading_string_matching_b200")
    for base, dirs, files in os.walk(pkg):
        dirs[:] = [d for d in dirs if d not in ("build", "bin", "__pycache__")]
        for f in files:
            if f.endswith((".py", ".c", ".h", ".cu", ".cuh")) or f == "Makefile":
                text = open(os.path.join(base, f), errors="replace").read()
                assert "oracle" not in text.lower(), os.path.join(base, f)
    ldd = subprocess.run(["ldd", kmp.LIB_PATH], capture_output=True, text=True).stdout
    assert "oracle" not in ldd


def test_pattern_loader_matches_oracle(oracle, strings_txt, tmp_path):
    assert kmp.load_patterns(strings_txt) == oracle.load_patterns(strings_txt)
    p = tmp_path / "s.txt"
    for content in (b"  foo\tbar\n\nfoo \x0b\x0c\r baz", b"", b"x" * 99 + b" ok\n", b"\xff\xfe \x01\x7f"):
        p.write_bytes(content)
        assert kmp.load_patterns(str(p)) == oracle.load_patterns(str(p))
    p.write_bytes(b"x" * 100)
    with pytest.raises(kmp.KmpbError) as e:
        kmp.load_patterns(str(p))
    assert e.value.code == -6
    p.write_bytes(b"ab\0cd")
    with pytest.raises(kmp.KmpbError):
        kmp.load_patterns(str(p))
    with pytest.raises(kmp.KmpbError) as e:
        kmp.load_patterns(str(tmp_path / "missing.txt"))
    assert e.value.code == -5


def test_extractors_match_reference_vectors(oracle):
    vectors = json.load(open(os.path.join(GOLDEN, "extract_vectors.json")))["vectors"]
    for v in vectors:
        frame = bytes.fromhex(v["frame"])
        got = kmp.extract_payload(frame, v["proto"])
        assert got == ((v["off"], v["len"]) if v["ok"] else None), v
        assert got == oracle.extract(frame, v["proto"])


@pytest.mark.parametrize("pcap", PCAPS)
@pytest.mark.parametrize("proto", ["udp", "tcp"])
def test_packer_matches_oracle_csr(oracle, pcap, proto):
    path = os.path.join(DATA, pcap + ".pcap")
    batch = kmp.PayloadBatch(path, proto, pinned=False)
    data, offsets, frames = oracle.load_pcap_csr(path, proto)
    assert (batch.n_frames, batch.n_packets, batch.total_bytes) == (frames, len(offsets) - 1, int(offsets[-1]))
    assert np.array_equal(batch.offsets, offsets)
    assert np.array_equal(batch.data, data)


def test_packer_savefile_variants(oracle, tmp_path):
    frames = [udp_frame(b"hello world"), b"short", udp_frame(b"", ihl=6), udp_frame(b"x" * 1400), udp_frame(b"a\0b")]
    want = None
    for name, kw in {"le_usec": {}, "le_nsec": {"magic": 0xA1B23C4D}, "be_usec": {"swapped": True},
                     "be_nsec": {"magic": 0xA1B23C4D, "swapped": True}}.items():
        p = str(tmp_path / (name + ".pcap"))
        write_pcap(p, frames, **kw)
        b = kmp.PayloadBatch(p, "udp")
        got = (b.n_frames, b.offsets.tolist(), b.data.tobytes())
        assert got[0] == 5 and got[1] == [0, 11, 11, 1411, 1414]
        assert want is None or got == want
        want = got
        d, o, fr = oracle.load_pcap_csr(p, "udp")
        assert (fr, o.tolist(), d.tobytes()) == got
    # a truncated trailing record ends the walk silently, like the reference's `>= 0` loop
    p = str(tmp_path / "trunc.pcap")
    write_pcap(p, frames)
    size = os.path.getsize(p)
    with open(p, "r+b") as f:
        f.truncate(size - 3)
    b = kmp.PayloadBatch(p, "udp")
    assert (b.n_frames, b.n_packets) == (4, 3)
    d, o, fr = oracle.load_pcap_csr(p, "udp")
    assert (fr, len(o) - 1) == (4, 3)
    # caplen < len: the captured bytes are what is parsed (openmp_data.c:114-116)
    p = str(tmp_path / "snap.pcap")
    write_pcap(p, [udp_frame(b"abcdefgh")], caplens=[46])
    b = kmp.PayloadBatch(p, "udp")
    assert b.data.tobytes() == b"abcd"
    # not a pcap
    (tmp_path / "bad.pcap").write_bytes(b"\0" * 64)
    with pytest.raises(kmp.KmpbError) as e:
        kmp.PayloadBatch(str(tmp_path / "bad.pcap"))
    assert e.value.code == -6
    with pytest.raises(kmp.KmpbError) as e:
        kmp.PayloadBatch(str(tmp_path / "nope.pcap"))
    assert e.value.code == -5


def test_savefile_payload_length_scan(tmp_path):
    """kmpb_pcap_first_long: the scan the savefile forms run over the accepted packets before anything else, to refuse
    a payload of KMPB_PACKET_LIMIT bytes or more (a payload is the captured length less the headers: any size)."""
    p = str(tmp_path / "lens.pcap")
    write_pcap(p, [udp_frame(b"x" * 10), b"not udp", udp_frame(b"y" * 300), udp_frame(b""), udp_frame(b"z" * 5000),
                    udp_frame(b"w" * 7)])
    lib = kmp.lib()
    fn = lib.kmpb_pcap_first_long
    fn.restype = ctypes.c_uint64
    fn.argtypes = [ctypes.c_void_p, ctypes.c_uint64, ctypes.c_uint64, ctypes.c_uint64]
    pc = ctypes.c_void_p()
    kmp.matcher.check(lib.kmpb_pcap_open(os.fsencode(p), kmp.PROTO_UDP, ctypes.byref(pc)))
    try:
        assert lib.kmpb_pcap_packets(pc) == 5  # payloads 10, 300, 0, 5000, 7
        assert fn(pc, 0, 5, 300) == 1
        assert fn(pc, 0, 5, 301) == 3
        assert fn(pc, 2, 3, 300) == 3
        assert fn(pc, 2, 1, 300) == 3  # none in [2, 3): first + count
        assert fn(pc, 4, 1, 8) == 5
        assert fn(pc, 4, 1, 7) == 4
        assert fn(pc, 0, 5, 5001) == 5
        assert fn(pc, 5, 0, 0) == 5
    finally:
        lib.kmpb_pcap_close(pc)


def test_packer_reads_pcapng(tmp_path):
    """SURVEY 8f-3: libpcap also hands the reference pcapng files; same frames, same batch."""
    frames = [udp_frame(b"hello world"), b"short", udp_frame(b"", ihl=6), udp_frame(b"x" * 1401), udp_frame(b"a\0b")]
    classic = str(tmp_path / "classic.pcap")
    write_pcap(classic, frames)
    b = kmp.PayloadBatch(classic, "udp")
    want = (b.n_frames, b.offsets.tolist(), b.data.tobytes())
    for name, kw in {"le": {}, "be": {"big_endian": True}, "simple": {"simple_from": 2},
                     "two_sections": {"second_section_at": 3}, "two_sections_be": {"big_endian": True, "second_section_at": 2}}.items():
        p = str(tmp_path / (name + ".pcapng"))
        with open(p, "wb") as f:
            f.write(pcapng(frames, **kw))
        b = kmp.PayloadBatch(p, "udp")
        assert (b.n_frames, b.offsets.tolist(), b.data.tobytes()) == want, name
    # a block cut short ends the walk silently
    p = str(tmp_path / "cut.pcapng")
    data = pcapng(frames)
    with open(p, "wb") as f:
        f.write(data[:-30])
    b = kmp.PayloadBatch(p, "udp")
    assert (b.n_frames, b.n_packets) == (4, 3)


def test_report_format(oracle):
    pats = [b"http", b"ack", b"zero", b"ack"]
    counts = [879, 8, 0, 8]
    assert kmp.format_report(pats, counts) == oracle.format_report(pats, counts)
    assert kmp.format_report([], []) == oracle.format_report([], [])


def test_shard_range_is_the_mpi_split():
    # mpi_dumping.c:149-157: N/P each, rank 0 also N%P, contiguous in rank order
    for n in (0, 1, 7, 8, 1000, 10_000_000):
        for world in (1, 2, 3, 4, 8):
            at = 0
            for rank in range(world):
                first, count = kmp.shard_range(n, world, rank)
                assert first == at and count == n // world + (n % world if rank == 0 else 0)
                at += count
            assert at == n


def test_synth_host_stream_properties():
    pats = kmp.load_patterns(os.path.join(DATA, "strings.txt"))
    s = kmp.Synth(seed=0xB200, payload_len=1400, plants=2, plant_patterns=pats)
    data, off = s.fill_host(0, 64)
    assert off.tolist() == [1400 * i for i in range(65)]
    pk = data.reshape(64, 1400)
    assert (pk[:, -1] == 0).all() and ((pk[:, :-1] >= 0x20) & (pk[:, :-1] <= 0x7E)).all()
    # slices of the stream are position independent
    d2, _ = s.fill_host(10, 5)
    assert np.array_equal(d2, data[14000:21000])
    # planted tokens are there
    assert sum(any(p in bytes(row) for p in set(pats)) for row in pk) == 64
    # mixed lengths (BASELINE config 5)
    m = kmp.Synth(seed=7, len_mode=1, plants=0)
    d, o = m.fill_host(0, 2000)
    lens = np.diff(o.astype(np.int64))
    assert set(lens.tolist()) == {64, 576, 1400, 9000}
    assert abs((lens == 64).mean() - 0.4) < 0.05 and abs((lens == 9000).mean() - 0.1) < 0.04
    assert m.nbytes(0, 2000) == int(o[-1]) and (d[o[1:].astype(np.int64) - 1] == 0).all()
    d3, o3 = m.fill_host(500, 100)
    assert np.array_equal(d3, d[int(o[500]):int(o[600])])


def test_host_tables_selfcheck(tmp_path):
    """tests/c/test_tables.c: union DFA == naive counts, prefilter never misses, NUL bit exact."""
    exe = str(tmp_path / "test_tables")
    subprocess.run(["/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc", "-O1", "-g", "-I" + os.path.join(ROOT, "include"),
                    "-I" + HOSTC, os.path.join(ROOT, "tests", "c", "test_tables.c"), os.path.join(HOSTC, "automaton.c"),
                    os.path.join(HOSTC, "errors.c"), "-o", exe], check=True)
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr


def test_cli_usage_and_errors(tmp_path):
    """serial.c:43,49,60-63: usage on stdout + exit 1; unreadable strings file -> perror + exit 1."""
    r = subprocess.run([MATCH], capture_output=True, text=True)
    assert r.returncode == 1 and r.stdout.startswith("USAGE: ") and "<file.pcap> <string.txt> [tcp/udp]" in r.stdout
    r = subprocess.run([MATCH, "a", "b", "icmp"], capture_output=True, text=True)
    assert r.returncode == 1 and r.stdout.startswith("USAGE ")
    r = subprocess.run([MATCH, "a", "b", "2", "icmp"], capture_output=True, text=True)
    assert r.returncode == 1 and "gpu_number" in r.stdout
    r = subprocess.run([MATCH, os.path.join(DATA, "udp.pcap"), str(tmp_path / "missing.txt")], capture_output=True, text=True)
    assert r.returncode == 1 and r.stderr.startswith("error opening file: ")


def test_bench_reference_arm_prints_one_contract_line():
    """`bench.py --impl reference` (runs on the host cores, no GPU): exactly one line on stdout, a JSON object with
    the keys the bench contract names for the reference arm."""
    import sys
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                        "--ref-packets", "1500"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "payload_GBps" and d["unit"] == "GB/s" and d["value"] > 0
    for key in ("n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data"):
        assert key in d, key
    assert d["dtype"] == "u8" and d["vs_baseline"] is None and "workload" in d["config"]
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["sample"]
    assert d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_bench_reference_arm_loads_no_product_code():
    """The reference arm must not run anything of the product: its sample comes from bench.py's numpy twin of the
    generator, which has to produce the very bytes of csrc/cuda/synth.cu, and libkmpb200.so is never mapped."""
    import importlib.util
    import sys
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    pats = kmp.load_patterns(os.path.join(DATA, "strings.txt"))
    assert bench.load_patterns_py(os.path.join(DATA, "strings.txt")) == pats
    for first, count, L in ((0, 700, 1400), (123457, 300, 1400), (5, 200, 64), (0, 40, 9000)):
        want, want_off = kmp.Synth(seed=bench.SEED, payload_len=L, plants=2, plant_patterns=pats).fill_host(first, count)
        got, got_off = bench.synth_stream(bench.SEED, first, count, L, 2, pats)
        assert np.array_equal(got, want) and np.array_equal(got_off, want_off)
    code = ("import sys; sys.argv=['bench.py','--impl','reference','--steps','1','--warmup','0','--ref-packets','600'];"
            "import runpy; runpy.run_path(%r, run_name='__main__');"
            "maps=open('/proc/self/maps').read(); sys.exit(3 if 'libkmpb200' in maps else 0)" % os.path.join(ROOT, "bench.py"))
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, (r.returncode, r.stderr[-1500:])


def test_host_side_is_sanitizer_clean(tmp_path):
    """The C host side (pattern loader, savefile reader, extractors, CSR packer, streamed packer, table builder,
    report) under AddressSanitizer + UndefinedBehaviorSanitizer over every bundled savefile and over damaged ones
    (truncated at many lengths, random bytes, empty).  The reference's own loader is not sanitizer-clean (SURVEY.md
    facts 9-11); ours has to be.  Known answers: SURVEY.md section 4."""
    exe = str(tmp_path / "test_host_sanitized")
    cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"
    srcs = [os.path.join(HOSTC, f) for f in ("errors.c", "extract.c", "patterns.c", "pcap_csr.c", "automaton.c")]
    subprocess.run([cc, "-O1", "-g", "-fsanitize=address,undefined", "-fno-sanitize-recover=all", "-fopenmp",
                    "-I" + os.path.join(ROOT, "include"), "-I" + HOSTC, os.path.join(ROOT, "tests", "c", "test_host_sanitized.c")]
                   + srcs + ["-o", exe], check=True)
    bundled = [os.path.join(DATA, f) for f in ("udp.pcap", "udp_1000.pcap", "big_udp.pcap", "very_big_udp.pcap", "tcp.pcap")]
    damaged = []
    whole = open(os.path.join(DATA, "udp_1000.pcap"), "rb").read()
    for i, cut in enumerate([0, 1, 23, 24, 25, 39, 40, 41, 100, 1000, len(whole) // 2, len(whole) - 1]):
        p = tmp_path / ("cut%d.pcap" % i)
        p.write_bytes(whole[:cut])
        damaged.append(str(p))
    rng = np.random.default_rng(5)
    (tmp_path / "noise.pcap").write_bytes(rng.integers(0, 256, 5000, dtype=np.uint8).tobytes())
    (tmp_path / "lying.pcap").write_bytes(whole[:24] + struct.pack("<IIII", 0, 0, 0xFFFFFFF0, 0xFFFFFFF0) + whole[40:400])
    damaged += [str(tmp_path / "noise.pcap"), str(tmp_path / "lying.pcap")]
    damaged += [str(tmp_path / "noise.pcap"), str(tmp_path / "lying.pcap")]
    # pcapng: both byte orders and several sections, whole and cut at every eighth byte, and with corrupted block lengths
    frames = [udp_frame(b"hello world"), b"short", udp_frame(b"", ihl=6), udp_frame(b"x" * 1401), udp_frame(b"a\0b")]
    for name, kw in {"le": {}, "be": {"big_endian": True}, "simple": {"simple_from": 2}, "two": {"second_section_at": 3}}.items():
        ng = pcapng(frames, **kw)
        for cut in list(range(0, min(len(ng), 400), 8)) + [len(ng) - 1, len(ng)]:
            p = tmp_path / ("%s_%d.pcapng" % (name, cut))
            p.write_bytes(ng[:cut])
            damaged.append(str(p))
        for at in (4, 32, 36, 60):
            bad = bytearray(ng)
            bad[at:at + 4] = b"\xff\xff\xff\x7f"
            p = tmp_path / ("%s_bad%d.pcapng" % (name, at))
            p.write_bytes(bytes(bad))
            damaged.append(str(p))
    env = dict(os.environ, ASAN_OPTIONS="detect_leaks=1:abort_on_error=0", UBSAN_OPTIONS="print_stacktrace=1", OMP_NUM_THREADS="4")
    r = subprocess.run([exe, os.path.join(DATA, "strings.txt")] + bundled + damaged, capture_output=True, text=True, env=env)
    assert r.returncode == 0, (r.stdout[-1500:], r.stderr[-3000:])
    for want in ("udp.pcap udp packets=20 bytes=3347 nulfree=11", "udp_1000.pcap udp packets=321 bytes=84519 nulfree=216",
                 "big_udp.pcap udp packets=3358 bytes=599424 nulfree=1038", "very_big_udp.pcap udp packets=13768 bytes=1321746 nulfree=0",
                 "tcp.pcap tcp packets=13 ", "udp_1000.pcap tcp packets=20 "):
        assert want in r.stdout, (want, r.stdout)


def test_integration_snippet_links_and_refuses_without_a_device(tmp_path):
    """The binding a maintainer of serial.c would write compiles warning-free against the public header alone; on a box
    without a B200 it stops at kmpb_create with the library's message instead of computing on the CPU."""
    r = subprocess.run([build_integration_snippet(tmp_path)], capture_output=True, text=True)
    if kmp.lib().kmpb_device_count() > 0:
        assert r.returncode == 0 and r.stdout == "aa: 3 times!\nhttp: 3 times!\n", (r.stdout, r.stderr)
    else:
        assert r.returncode == 1 and "no CPU path" in r.stderr and r.stdout == "", (r.stdout, r.stderr)
