"""Which packets match: kmpb_select_* (the union engine's mark kernel, the verdict and compaction passes), the savefile
writer kmpb_pcap_write_selected, Matcher.select_*, kmp.write_selected and bin/kmp_select.

A packet is selected iff it holds at least one match the count forms count: exactly the packets the reference finder
(tests/c/kmp_find_ref.c) reports a record for.  The CPU tests check the writer on hand-built savefiles of every kind the
reader takes, the writer on the bundled captures with the reference finder's verdicts, the entry points without a
device, and that the existing union kernels compile to the same SASS as before the mark kernel was added.  The GPU
tests check every select form against the reference finder (case-sensitive sets) or the find forms (nocase sets)."""
import ctypes
import hashlib
import json
import os
import re
import struct
import subprocess

import numpy as np
import pytest

from conftest import DATA, GOLDEN, ROOT
from test_find import RefFinder, csr, pcap_frames
from test_host import _pcapng, _udp_frame, _write_pcap

import multithreading_string_matching_b200 as kmp

PKG = os.path.join(ROOT, "multithreading_string_matching_b200")
SELECT = os.path.join(PKG, "bin", "kmp_select")
MATCH = os.path.join(PKG, "bin", "kmp_match")
PCAPS = ["udp", "udp_1000", "big_udp", "very_big_udp", "tcp"]
EINVAL, ESTATE = -1, -7


@pytest.fixture(scope="module")
def finder(tmp_path_factory):
    return RefFinder(str(tmp_path_factory.mktemp("kmp_find_ref_sel")))


def expected_flags(finder, data, offsets, patterns):
    """the packets with at least one record of the reference finder"""
    n = len(offsets) - 1
    flags = np.zeros(n, dtype=bool)
    if patterns and n:
        flags[finder.find_csr(data, offsets, patterns)["packet"].astype(np.int64)] = True
    return flags


# ---- savefile parsing for the checks --------------------------------------------------------------------

def classic_records(path):
    """(global header, [whole record bytes]) of a classic savefile, up to a cut trailing record"""
    raw = open(path, "rb").read()
    e = "<" if struct.unpack("<I", raw[:4])[0] in (0xA1B2C3D4, 0xA1B23C4D) else ">"
    at, recs = 24, []
    while len(raw) - at >= 16:
        cap = struct.unpack(e + "I", raw[at + 8:at + 12])[0]
        if cap > len(raw) - at - 16:
            break
        recs.append(raw[at:at + 16 + cap])
        at += 16 + cap
    return raw[:24], recs


def pcapng_blocks(raw):
    """[(is_packet_block, block bytes)] of a well-formed pcapng file"""
    at, out, e = 0, [], "<"
    while len(raw) - at >= 12:
        if raw[at:at + 4] == b"\x0a\x0d\x0d\x0a":
            e = "<" if struct.unpack("<I", raw[at + 8:at + 12])[0] == 0x1A2B3C4D else ">"
        btype, total = struct.unpack(e + "II", raw[at:at + 8])
        out.append((btype in (2, 3, 6), raw[at:at + total]))
        at += total
    return out


def open_pcap(path, proto="udp"):
    lib = kmp.lib()
    pc = ctypes.c_void_p()
    kmp.matcher.check(lib.kmpb_pcap_open(os.fsencode(path), kmp.matcher._PROTO[proto], ctypes.byref(pc)))
    return pc


def accepted_frames(path, proto="udp"):
    lib = kmp.lib()
    pc = open_pcap(path, proto)
    try:
        n = lib.kmpb_pcap_packets(pc)
        frames = np.zeros(max(n, 1), dtype=np.uint64)
        kmp.matcher.check(lib.kmpb_pcap_frame_index(pc, 0, n, frames.ctypes.data))
        return frames[:n].astype(np.int64)
    finally:
        lib.kmpb_pcap_close(pc)


def _pb_pcapng(frames, big_endian=False):
    """SHB, IDB, then obsolete Packet Blocks (type 2) and an Interface Statistics Block at the end"""
    e = ">" if big_endian else "<"

    def block(btype, body):
        body += b"\0" * (-len(body) % 4)
        return struct.pack(e + "II", btype, len(body) + 12) + body + struct.pack(e + "I", len(body) + 12)

    out = block(0x0A0D0D0A, struct.pack(e + "IHHq", 0x1A2B3C4D, 1, 0, -1))
    out += block(1, struct.pack(e + "HHI", 1, 0, 65535))
    for k, f in enumerate(frames):
        out += block(2, struct.pack(e + "HHIIII", 0, 0, 0, k, len(f), len(f)) + f)
    return out + block(5, struct.pack(e + "III", 0, 0, 0))


FRAMES = [_udp_frame(b"hello world"), b"short", _udp_frame(b"", ihl=6), _udp_frame(b"x" * 1400), _udp_frame(b"a\0b"),
          _udp_frame(b"ack ack"), _udp_frame(b"z" * 77)]


def check_written(src, flags, tmp_path, tag):
    """write_selected with flags and inverted: each output holds exactly its chosen records, verbatim and in order, and
    the two partition the accepted frames; a re-opened output has the chosen packets; all-false: no packet at all"""
    acc = accepted_frames(src)
    flags = np.asarray(flags, dtype=bool)
    assert len(flags) == len(acc)
    raw = open(src, "rb").read()
    outs = {}
    for inv in (False, True):
        out = str(tmp_path / ("%s_%d" % (tag, inv)))
        n = kmp.write_selected(src, "udp", flags, out, invert=inv)
        chosen = acc[flags != inv]
        assert n == len(chosen), (tag, inv)
        b = kmp.PayloadBatch(out, "udp")
        assert b.n_packets == len(chosen) and b.n_frames == len(chosen), (tag, inv)
        outs[inv] = (out, chosen)
    if raw[:4] == b"\x0a\x0d\x0d\x0a":
        blocks = pcapng_blocks(raw)
        packets = [blk for is_p, blk in blocks if is_p]
        for inv, (out, chosen) in outs.items():
            keep = set(chosen.tolist())
            frame, want = 0, []
            for is_p, blk in blocks:
                if is_p:
                    if frame in keep:
                        want.append(blk)
                    frame += 1
                else:
                    want.append(blk)
            assert open(out, "rb").read() == b"".join(want), (tag, inv)
        assert len(packets) >= len(acc)
    else:
        hdr, recs = classic_records(src)
        for inv, (out, chosen) in outs.items():
            ohdr, orecs = classic_records(out)
            assert ohdr == hdr and orecs == [recs[f] for f in chosen.tolist()], (tag, inv)
            assert open(out, "rb").read() == hdr + b"".join(orecs)
    # the partition, in order: merging by frame number gives back every accepted frame once
    both = sorted(outs[False][1].tolist() + outs[True][1].tolist())
    assert both == acc.tolist()


# ---- CPU ------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("variant", ["le_usec", "le_nsec", "be_usec", "be_nsec", "snaplen", "cut_tail"])
def test_writer_classic(tmp_path, variant):
    kw = {"le_usec": {}, "le_nsec": {"magic": 0xA1B23C4D}, "be_usec": {"swapped": True},
          "be_nsec": {"magic": 0xA1B23C4D, "swapped": True}, "snaplen": {}, "cut_tail": {}}[variant]
    caplens = None
    if variant == "snaplen":  # caplen < len records are kept as they are
        caplens = [len(f) if i % 2 else min(len(f), 46) for i, f in enumerate(FRAMES)]
    src = str(tmp_path / "in.pcap")
    _write_pcap(src, FRAMES, caplens=caplens, **kw)
    if variant == "cut_tail":
        with open(src, "r+b") as f:
            f.truncate(os.path.getsize(src) - 20)
    n = len(accepted_frames(src))
    rng = np.random.default_rng(7)
    for i, flags in enumerate([rng.random(n) < 0.5, np.ones(n, bool), np.zeros(n, bool), np.arange(n) % 2 == 1]):
        check_written(src, flags, tmp_path, "%s%d" % (variant, i))
    # all-false: a header-only file
    out = str(tmp_path / "none.pcap")
    assert kmp.write_selected(src, "udp", np.zeros(n, bool), out) == 0
    assert open(out, "rb").read() == open(src, "rb").read()[:24]


@pytest.mark.parametrize("variant", ["le", "be", "simple", "two_sections", "two_sections_be", "packet_blocks",
                                     "packet_blocks_be"])
def test_writer_pcapng(tmp_path, variant):
    if variant.startswith("packet_blocks"):
        raw = _pb_pcapng(FRAMES, big_endian=variant.endswith("_be"))
    else:
        kw = {"le": {}, "be": {"big_endian": True}, "simple": {"simple_from": 2}, "two_sections": {"second_section_at": 3},
              "two_sections_be": {"big_endian": True, "second_section_at": 2}}[variant]
        raw = _pcapng(FRAMES, **kw)
    src = str(tmp_path / "in.pcapng")
    open(src, "wb").write(raw)
    n = len(accepted_frames(src))
    assert n == 6
    rng = np.random.default_rng(11)
    for i, flags in enumerate([rng.random(n) < 0.5, np.ones(n, bool), np.zeros(n, bool), np.arange(n) % 2 == 0]):
        check_written(src, flags, tmp_path, "%s%d" % (variant, i))
    out = str(tmp_path / "none.pcapng")
    assert kmp.write_selected(src, "udp", np.zeros(n, bool), out) == 0
    assert all(not is_p for is_p, _ in pcapng_blocks(open(out, "rb").read()))


def test_writer_section_length_is_unspecified(tmp_path):
    """A section header that declares its length is written with -1 (not specified): the written section is shorter.
    Every other byte of every kept block is the input's."""
    for big in (False, True):
        e = ">" if big else "<"
        raw = bytearray(_pcapng(FRAMES, big_endian=big, second_section_at=3))
        shbs = [at for at in range(0, len(raw), 4) if raw[at:at + 4] == b"\x0a\x0d\x0d\x0a"]
        assert len(shbs) == 2
        ends = shbs[1:] + [len(raw)]
        for at, end in zip(shbs, ends):  # the section's length after its header block
            e_at = "<" if struct.unpack("<I", raw[at + 8:at + 12])[0] == 0x1A2B3C4D else ">"
            total = struct.unpack(e_at + "I", raw[at + 4:at + 8])[0]
            raw[at + 16:at + 24] = struct.pack(e_at + "q", end - at - total)
        src = str(tmp_path / ("len_%d.pcapng" % big))
        open(src, "wb").write(bytes(raw))
        n = len(accepted_frames(src))
        flags = np.arange(n) % 2 == 0
        out = str(tmp_path / ("out_%d.pcapng" % big))
        kmp.write_selected(src, "udp", flags, out)
        got = pcapng_blocks(open(out, "rb").read())
        chosen, frame, want = set(accepted_frames(src)[flags].tolist()), 0, []
        for is_p, blk in pcapng_blocks(bytes(raw)):
            if is_p:
                if frame in chosen:
                    want.append(blk)
                frame += 1
            elif blk[:4] == b"\x0a\x0d\x0d\x0a":
                want.append(blk[:16] + b"\xff" * 8 + blk[24:])
            else:
                want.append(blk)
        assert [blk for _, blk in got] == want, big
        assert kmp.PayloadBatch(out, "udp").n_packets == int(flags.sum())


def test_writer_slices_and_refusals(tmp_path):
    src = str(tmp_path / "in.pcap")
    _write_pcap(src, FRAMES)
    acc = accepted_frames(src)
    _, recs = classic_records(src)
    out = str(tmp_path / "out.pcap")
    # first / count: the flags are those of accepted packets [first, first + count)
    assert kmp.write_selected(src, "udp", [True, False, True], out, first=1) == 2
    assert classic_records(out)[1] == [recs[acc[1]], recs[acc[3]]]
    assert kmp.write_selected(src, "udp", [True, False, True], out, first=1, invert=True) == 1
    assert classic_records(out)[1] == [recs[acc[2]]]
    with pytest.raises(kmp.KmpbError) as e:
        kmp.write_selected(src, "udp", [True] * 3, out, first=len(acc) - 2)
    assert e.value.code == EINVAL
    # the input itself, by its own name, another path and a hard link: refused, the input intact
    before = open(src, "rb").read()
    link = str(tmp_path / "link.pcap")
    os.link(src, link)
    for path in (src, str(tmp_path / "." / "in.pcap"), link):
        with pytest.raises(kmp.KmpbError) as e:
            kmp.write_selected(src, "udp", np.ones(len(acc), bool), path)
        assert e.value.code == EINVAL and "input savefile" in str(e.value)
    assert open(src, "rb").read() == before
    # an unwritable place: KMPB_EIO, nothing left behind
    with pytest.raises(kmp.KmpbError) as e:
        kmp.write_selected(src, "udp", np.ones(len(acc), bool), str(tmp_path / "no" / "such" / "dir.pcap"))
    assert e.value.code == -5


@pytest.mark.parametrize("pcap", PCAPS)
@pytest.mark.parametrize("proto", ["udp", "tcp"])
def test_expected_verdicts_write_the_matching_frames(oracle, finder, strings_txt, tmp_path, pcap, proto):
    """The reference finder's verdicts on the bundled captures, written out: the selected frames hold every match of
    the input (same counts), the others none."""
    path = os.path.join(DATA, pcap + ".pcap")
    pats = kmp.load_patterns(strings_txt)
    b = kmp.PayloadBatch(path, proto)
    flags = expected_flags(finder, b.data, b.offsets, pats)
    want = oracle.count_csr(b.data, b.offsets, pats)
    for inv in (False, True):
        out = str(tmp_path / ("out_%d.pcap" % inv))
        assert kmp.write_selected(path, proto, flags, out, invert=inv) == int((flags != inv).sum())
        o = kmp.PayloadBatch(out, proto)
        got = oracle.count_csr(o.data, o.offsets, pats)
        assert got == (want if not inv else [0] * len(pats)), (pcap, proto, inv)


def test_select_needs_a_device(tmp_path):
    """No CPU path: the select entry points refuse a NULL context, kmp_select stops with kmp_find's message."""
    import torch

    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    lib = kmp.lib()
    n = ctypes.c_uint64(0)
    flags = (ctypes.c_uint8 * 4)()
    assert lib.kmpb_select_host(None, None, None, 0, flags, ctypes.byref(n), None) == EINVAL
    assert lib.kmpb_select_pcap(None, None, 0, 0, flags, ctypes.byref(n), None) == EINVAL
    assert lib.kmpb_select_device_span(None, None, None, 0, 0, 0, None, None, None, None, 0, None) == EINVAL
    out = str(tmp_path / "out.pcap")
    r = subprocess.run([SELECT, os.path.join(DATA, "udp.pcap"), os.path.join(DATA, "strings.txt"), out],
                       capture_output=True, text=True)
    assert r.returncode == 1 and "no CPU path" in r.stderr and r.stdout == "" and not os.path.exists(out)


def test_kmp_select_usage_and_errors(tmp_path):
    usage = "USAGE: ./kmp_select [-i] [-v] <file.pcap> <string.txt> <out.pcap> [tcp/udp]\n"
    for args in ([], ["a", "b"], ["-i", "-v", "a", "b"]):
        r = subprocess.run([SELECT] + args, capture_output=True, text=True)
        assert r.returncode == 1 and r.stdout == usage, args
    r = subprocess.run([SELECT, "a", "b", "c", "icmp"], capture_output=True, text=True)
    assert r.returncode == 1 and r.stdout.startswith("USAGE ")
    r = subprocess.run([SELECT, os.path.join(DATA, "udp.pcap"), str(tmp_path / "missing.txt"), str(tmp_path / "o")],
                       capture_output=True, text=True)
    assert r.returncode == 1 and r.stderr.startswith("error opening file: ")


def _sass_by_kernel(obj):
    sass = subprocess.run([os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "cuobjdump"), "-sass", obj],
                          capture_output=True, text=True, check=True).stdout
    out, cur = {}, None
    for line in sass.splitlines(keepends=True):
        m = re.search(r"Function : (\S+)", line)
        if m:
            cur = m.group(1)
            out[cur] = []
        elif cur:
            out[cur].append(line)
    return {k: "".join(v) for k, v in out.items()}


def test_existing_union_kernels_compile_to_the_same_sass():
    """The count and find kernels (and their nocase twins) are the same machine code as before the mark kernel was
    added: tests/golden/union_sass_sha256.json holds the SHA-256 of each one's `cuobjdump -sass` listing, built with the
    Makefile's flags by the nvcc named there."""
    golden = json.load(open(os.path.join(GOLDEN, "union_sass_sha256.json")))
    nvcc = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "nvcc")
    obj = os.path.join(PKG, "build", "union_kernel.o")
    if not os.path.exists(obj) or not os.path.exists(nvcc):
        pytest.skip("no union_kernel.o or no nvcc")
    version = subprocess.run([nvcc, "--version"], capture_output=True, text=True).stdout.strip().splitlines()[-1]
    if version != golden["nvcc"]:
        pytest.skip("the hashes are of %s, this is %s" % (golden["nvcc"], version))
    sass = _sass_by_kernel(obj)
    for name, digest in golden["sha256"].items():
        assert hashlib.sha256(sass[name].encode()).hexdigest() == digest, name
    assert "_Z22kmpb_union_mark_kernel12union_paramsPj" in sass and "_Z29kmpb_union_mark_nocase_kernel12union_paramsPj" in sass


# ---- GPU ------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def matcher():
    m = kmp.Matcher(0)
    yield m
    m.close()


@pytest.fixture(scope="module")
def strings(strings_txt):
    return kmp.load_patterns(strings_txt)


def device_select(m, data, offsets, k0=0, k1=None, invert=False, stream=None, sync=True, n_pat=None):
    """kmpb_select_device_span over packets [k0, k1) of a device copy of the batch -> (flags, index list, counts);
    the counts start at 5 each (accumulated into)."""
    import torch

    k1 = len(offsets) - 1 if k1 is None else k1
    n = k1 - k0
    n_pat = len(m.patterns) if n_pat is None else n_pat
    d_bytes = torch.zeros(((len(data) + 64 + 31) // 32) * 32, dtype=torch.uint8, device="cuda:0")
    if len(data):
        d_bytes[: len(data)] = torch.from_numpy(np.array(data, dtype=np.uint8)).cuda()
    d_off = torch.from_numpy(np.ascontiguousarray(offsets, dtype=np.int64)).cuda()
    d_flags = torch.full((max(n, 1),), 7, dtype=torch.uint8, device="cuda:0")
    d_index = torch.full((max(n, 1),), -1, dtype=torch.int64, device="cuda:0")
    d_n = torch.full((1,), -1, dtype=torch.int64, device="cuda:0")
    d_counts = torch.full((max(n_pat, 1),), 5, dtype=torch.int64, device="cuda:0")
    span = (int(offsets[k0]), int(offsets[k1]))
    m.select_device(d_bytes.data_ptr(), d_off.data_ptr() + 8 * k0, n, d_flags.data_ptr(), span, d_index.data_ptr(),
                    d_n.data_ptr(), d_counts.data_ptr(), invert=invert, stream=stream)
    res = lambda: (d_flags[:n].cpu().numpy().astype(bool), d_index[: int(d_n.item())].cpu().numpy(),  # noqa: E731
                   [c - 5 for c in d_counts[:n_pat].cpu().tolist()])
    if sync:
        torch.cuda.synchronize()
        return res()
    return res, (d_bytes, d_off, d_flags, d_index, d_n, d_counts)


def check_batch(m, data, offsets, want, label=""):
    """host and device forms (plain and inverted) against the expected verdicts; counts against kmpb_count_host"""
    n = len(offsets) - 1
    flags, counts = m.select_host(data, offsets)
    assert np.array_equal(flags, want), (label, "host", np.flatnonzero(flags != want)[:8])
    want_counts = m.count_host(data, offsets) if m.patterns else []
    assert counts == want_counts, (label, "host counts")
    for inv in (False, True):
        f, idx, c = device_select(m, data, offsets, invert=inv)
        assert np.array_equal(f, want), (label, "device", inv, np.flatnonzero(f != want)[:8])
        assert np.array_equal(idx, np.flatnonzero(want != inv)), (label, "index", inv)
        assert c == want_counts, (label, "device counts")
    assert len(want) == n
    # *n_selected of the host form, and the form without counts_out
    d = np.array(data, dtype=np.uint8) if len(data) else np.zeros(1, np.uint8)
    o = np.ascontiguousarray(offsets, dtype=np.uint64)
    fl = np.zeros(max(n, 1), dtype=np.uint8)
    n_sel = ctypes.c_uint64(12345)
    kmp.matcher.check(kmp.lib().kmpb_select_host(m.handle, d.ctypes.data, o.ctypes.data, n, fl.ctypes.data,
                                                 ctypes.byref(n_sel), None))
    assert n_sel.value == int(want.sum()) and np.array_equal(fl[:n].astype(bool), want), (label, "n_selected")
    kmp.matcher.check(kmp.lib().kmpb_check_device_errors(m.handle))


@pytest.mark.gpu
@pytest.mark.parametrize("pcap", PCAPS)
@pytest.mark.parametrize("proto", ["udp", "tcp"])
@pytest.mark.parametrize("nocase", [False, True])
def test_bundled_captures(matcher, finder, strings, pcap, proto, nocase):
    path = os.path.join(DATA, pcap + ".pcap")
    matcher.set_patterns(strings, nocase=nocase)
    b = kmp.PayloadBatch(path, proto)
    if nocase:  # the find forms' packets (their records are checked against the reference in test_nocase.py)
        want = np.zeros(b.n_packets, dtype=bool)
        want[matcher.find_host(b.data, b.offsets)["packet"].astype(np.int64)] = True
    else:
        want = expected_flags(finder, b.data, b.offsets, strings)
    check_batch(matcher, b.data, b.offsets, want, (pcap, proto, nocase))
    assert np.array_equal(matcher.select_pcap(path, proto), want)
    n = b.n_packets
    if n > 4:
        assert np.array_equal(matcher.select_pcap(path, proto, 1, n - 3), want[1:n - 2])


def silence(data, offsets, every=2):
    """a copy of the batch in which every `every`-th packet holds only 0x01 bytes (no pattern of strings.txt)"""
    data = np.array(data, dtype=np.uint8)
    for k in range(0, len(offsets) - 1, every):
        data[int(offsets[k]):int(offsets[k + 1])] = 1
    return data


def distinct_total(counts, patterns):
    """the number of find records: every distinct pattern's count once"""
    seen = set()
    return sum(c for c, p in zip(counts, patterns) if not (p in seen or seen.add(p)))


def _uniform(n, size, fill):
    return [fill * size for _ in range(n)]


@pytest.mark.gpu
def test_edge_batches(matcher, finder):
    rng = np.random.default_rng(5)
    p99 = bytes(rng.integers(97, 100, 99).astype(np.uint8))
    cases = {
        "nul_before_only_match": ([b"xx\0http", b"http", b"ht\0tp"], [b"http"]),
        "match_ends_packet": ([b"xxhttp", b"xhtt", b"p", b"http"], [b"http", b"p"]),
        "empty_and_one_byte": ([b"", b"a", b"", b"", b"b", b"a", b""] + [b""] * 500 + [b"a"], [b"a"]),
        "long_empty_runs": ([b""] * 3000 + [b"zz"] + [b""] * 5000 + [b"az"], [b"az", b"z"]),
        "lengths_1_2_9_99": ([b"q" + p99 + b"q", p99[:50], b"abcdefghi", b"ab", b"c"], [b"c", b"ab", b"abcdefghi", p99]),
        "uniform_size": (_uniform(4096, 64, b"k") + [b"x" * 64], [b"x"]),
        "uniform_with_matches": ([bytes(rng.integers(97, 101, 96).astype(np.uint8)) for _ in range(3000)], [b"abc", b"dd"]),
        "dense_one_byte": ([b"a" * int(s) for s in rng.integers(0, 3, 20000)], [b"a"]),
        "dense_many_packets_per_word": ([b"ab"[int(x)] .to_bytes(1, "little") * int(s) for x, s in
                                         zip(rng.integers(0, 2, 30000), rng.integers(0, 4, 30000))], [b"b"]),
        "no_patterns": ([b"abc", b"def"], []),
        "empty_batch": ([], [b"a"]),
        "all_empty_packets": ([b""] * 77, [b"a"]),
    }
    for label, (pkts, pats) in cases.items():
        matcher.set_patterns(pats)
        data, offsets = csr(pkts)
        check_batch(matcher, data, offsets, expected_flags(finder, data, offsets, pats), label)


@pytest.mark.gpu
def test_first_byte_not_a_multiple_of_32(matcher, finder):
    """device spans and host batches that start at every residue of 32 (offsets relative to absolute byte 0)"""
    rng = np.random.default_rng(9)
    pats = [b"ab", b"b", b"abcab", b"cc"]
    matcher.set_patterns(pats)
    pkts = [bytes(rng.integers(97, 100, int(s)).astype(np.uint8)) for s in rng.integers(0, 40, 4000)]
    data, offsets = csr(pkts)
    want = expected_flags(finder, data, offsets, pats)
    seen = set()
    for k0 in range(0, 400):
        if int(offsets[k0]) % 32 in seen:
            continue
        seen.add(int(offsets[k0]) % 32)
        k1 = len(pkts) - int(rng.integers(0, 50))
        f, idx, c = device_select(matcher, data, offsets, k0, k1)
        assert np.array_equal(f, want[k0:k1]), k0
        assert np.array_equal(idx, np.flatnonzero(want[k0:k1]))
        sub = offsets[k0:k1 + 1]
        flags, counts = matcher.select_host(data, sub)
        assert np.array_equal(flags, want[k0:k1]) and counts == matcher.count_host(data, sub), k0
    assert len(seen) >= 16


@pytest.mark.gpu
def test_random_batches_and_global_tables(finder):
    rng = np.random.default_rng(1234)
    with kmp.Matcher(0) as m:
        for trial in range(12):
            alpha = [b"ab", b"ab\0", b"abcd", bytes(range(1, 256))][trial % 4]
            pats = [bytes(rng.choice(list(alpha.replace(b"\0", b""))) for _ in range(int(rng.choice([1, 2, 3, 5, 9, 99]))))
                    for _ in range(int(rng.integers(1, 9)))]
            pkts = [bytes(rng.choice(list(alpha), int(s)).astype(np.uint8)) for s in rng.choice([0, 1, 3, 17, 120, 1400], 3000)]
            m.set_patterns(pats)
            data, offsets = csr(pkts)
            check_batch(m, data, offsets, expected_flags(finder, data, offsets, pats), ("random", trial))
        # ~800 patterns: the probe tables leave shared memory
        pkts = [bytes(rng.integers(97, 105, int(s)).astype(np.uint8)) for s in rng.integers(0, 600, 6000)]
        data, offsets = csr(pkts)
        pats = []
        while len(pats) < 800:
            p = pkts[int(rng.integers(0, len(pkts)))]
            ln = int(rng.choice([2, 3, 4, 5, 9, 17, 40]))
            if len(p) > ln:
                at = int(rng.integers(0, len(p) - ln))
                pats.append(p[at:at + ln] if rng.random() < 0.3 else bytes(rng.integers(97, 105, ln).astype(np.uint8)))
        m.set_patterns(pats)
        check_batch(m, data, offsets, expected_flags(finder, data, offsets, pats), "global tables")


@pytest.mark.gpu
def test_chunked_forms(monkeypatch, finder, strings):
    """1 MiB chunks: many chunks through every stream slot, host and savefile forms, first / count slices"""
    monkeypatch.setenv("KMPB_CHUNK_MB", "1")
    synth = kmp.Synth(seed=77, payload_len=1400, len_mode=1, plants=1, plant_patterns=strings)
    data, offsets = synth.fill_host(0, 12000)
    data = silence(data, offsets, 3)
    with kmp.Matcher(0) as m:
        m.set_patterns(strings)
        want = expected_flags(finder, data, offsets, strings)
        assert 0 < want.sum() < len(want)
        flags, counts = m.select_host(data, offsets)
        assert np.array_equal(flags, want) and counts == m.count_host(data, offsets)
        path = os.path.join(DATA, "very_big_udp.pcap")
        b = kmp.PayloadBatch(path, "udp")
        pw = expected_flags(finder, b.data, b.offsets, strings)
        n = b.n_packets
        for first, count in ((0, n), (1, n - 1), (n // 3, n // 2), (n - 1, 1), (5, 0)):
            assert np.array_equal(m.select_pcap(path, "udp", first, count), pw[first:first + count]), (first, count)


@pytest.mark.gpu
def test_back_to_back_selects_are_independent(matcher, finder, strings):
    """a verdict pass that left bits behind would select packets of the previous batch"""
    matcher.set_patterns(strings)
    synth = kmp.Synth(seed=3, payload_len=700, plants=1, plant_patterns=strings)
    data_a, off_a = synth.fill_host(0, 5000)
    data_a = silence(data_a, off_a, 2)
    data_b, off_b = synth.fill_host(5000, 4000)
    data_b = silence(data_b, off_b, 5)
    want_a = expected_flags(finder, data_a, off_a, strings)
    want_b = expected_flags(finder, data_b, off_b, strings)
    assert want_a.any() and not want_a.all() and not np.array_equal(want_a[:4000], want_b)
    for _ in range(2):
        for data, off, want in ((data_a, off_a, want_a), (data_b, off_b, want_b), (data_a, off_a, want_a)):
            assert np.array_equal(device_select(matcher, data, off)[0], want)
            assert np.array_equal(matcher.select_host(data, off)[0], want)


@pytest.mark.gpu
def test_interleaved_with_count_and_find(finder, strings):
    """selects, counts and finds on three streams with no host sync in between give the answers each gives alone;
    KMPB_ESTATE while a frame stream is open"""
    import torch

    synth = kmp.Synth(seed=21, payload_len=900, len_mode=1, plants=2, plant_patterns=strings)
    data, offsets = synth.fill_host(0, 20000)
    want = expected_flags(finder, data, offsets, strings)
    with kmp.Matcher(0) as m:
        m.set_patterns(strings)
        want_counts = m.count_host(data, offsets)
        total = distinct_total(want_counts, strings)
        streams = [torch.cuda.Stream() for _ in range(3)]
        keep, results = [], []
        d_bytes = torch.from_numpy(np.concatenate([data, np.zeros(64, np.uint8)])).cuda()
        d_off = torch.from_numpy(offsets.astype(np.int64)).cuda()
        torch.cuda.synchronize()
        span = (0, int(offsets[-1]))
        n = len(offsets) - 1
        for rnd in range(3):
            res, bufs = device_select(m, data, offsets, stream=streams[0].cuda_stream, sync=False)
            keep.append(bufs)
            results.append(res)
            d_counts = torch.zeros(len(strings), dtype=torch.int64, device="cuda:0")
            m.count_device(d_bytes.data_ptr(), d_off.data_ptr(), n, d_counts.data_ptr(), span=span, stream=streams[1].cuda_stream)
            d_rec = torch.zeros(total * 16, dtype=torch.uint8, device="cuda:0")
            d_n = torch.zeros(1, dtype=torch.int64, device="cuda:0")
            m.find_device(d_bytes.data_ptr(), d_off.data_ptr(), n, d_rec.data_ptr(), total, d_n.data_ptr(), span,
                          stream=streams[2].cuda_stream)
            keep.append((d_counts, d_rec, d_n))
        torch.cuda.synchronize()
        for res in results:
            f, idx, c = res()
            assert np.array_equal(f, want) and np.array_equal(idx, np.flatnonzero(want)) and c == want_counts
        for d_counts, d_rec, d_n in keep[1::2]:
            assert d_counts.cpu().tolist() == want_counts and int(d_n.item()) == total
            pk = np.unique(d_rec.cpu().numpy().view(kmp.MATCH_DTYPE)["packet"].astype(np.int64))
            assert np.array_equal(pk, np.flatnonzero(want))
        with m.stream("udp") as st:
            st.push(_udp_frame(b"x"))
            for call in (lambda: m.select_host(data, offsets), lambda: device_select(m, data, offsets),
                         lambda: m.select_pcap(os.path.join(DATA, "udp.pcap"))):
                with pytest.raises(kmp.KmpbError) as e:
                    call()
                assert e.value.code == ESTATE
        assert np.array_equal(m.select_host(data, offsets)[0], want)


@pytest.mark.gpu
def test_first_select_and_growth_on_a_side_stream(strings):
    """A fresh context's first device select, and one whose batch grows the bitmap, on a non-blocking side stream with
    no host sync before it: the bitmap is zeroed on that stream, ahead of the mark kernel (a zeroing on another stream
    could wipe bits the kernel had set).  Verdicts against the packets of the find records."""
    import torch

    synth = kmp.Synth(seed=0x5E1, payload_len=1400, plants=1, plant_patterns=strings)
    n_all = 1_200_000
    nbytes = synth.nbytes(0, n_all)
    with kmp.Matcher(0) as m:
        m.set_patterns(strings)
        d_bytes = torch.empty(nbytes + 4096, dtype=torch.uint8, device="cuda:0")
        d_off = torch.empty(n_all + 1, dtype=torch.int64, device="cuda:0")
        synth.fill_device(m, 0, n_all, d_bytes.data_ptr(), d_off.data_ptr())
        d_bytes[: n_all * 1400].view(n_all, 1400)[::3] = 1  # every third packet without a match
        off = d_off.cpu().numpy()
        wants = {}
        for n in (300_000, n_all):  # the second grows the bitmap
            counts = torch.zeros(len(strings), dtype=torch.int64, device="cuda:0")
            m.count_device(d_bytes.data_ptr(), d_off.data_ptr(), n, counts.data_ptr(), span=(0, int(off[n])))
            torch.cuda.synchronize()
            total = distinct_total(counts.cpu().tolist(), strings)
            d_rec = torch.empty(total * 16, dtype=torch.uint8, device="cuda:0")
            d_n = torch.zeros(1, dtype=torch.int64, device="cuda:0")
            m.find_device(d_bytes.data_ptr(), d_off.data_ptr(), n, d_rec.data_ptr(), total, d_n.data_ptr(), (0, int(off[n])))
            torch.cuda.synchronize()
            w = np.zeros(n, dtype=bool)
            w[d_rec.cpu().numpy().view(kmp.MATCH_DTYPE)["packet"].astype(np.int64)] = True
            wants[n] = w
    for order in ((300_000, n_all), (n_all,)):
        with kmp.Matcher(0) as m:
            m.set_patterns(strings)
            side = torch.cuda.Stream()
            for n in order:
                d_flags = torch.empty(n, dtype=torch.uint8, device="cuda:0")
                torch.cuda.synchronize()
                m.select_device(d_bytes.data_ptr(), d_off.data_ptr(), n, d_flags.data_ptr(), (0, int(off[n])),
                                stream=side.cuda_stream)
                side.synchronize()
                got = d_flags.cpu().numpy().astype(bool)
                assert np.array_equal(got, wants[n]), (order, n, np.flatnonzero(got != wants[n])[:8])
                assert 0 < got.sum() < n


@pytest.mark.gpu
def test_device_batch_past_4GiB(strings):
    """~4.6 GB of synthetic traffic on the device, a span from an odd first byte across 2^32: the verdicts are the
    packets of that span's find records, the counts those of the count form"""
    import torch

    free, _ = torch.cuda.mem_get_info()
    if free < 12 * 2**30:
        pytest.skip("needs 12 GiB of device memory")
    synth = kmp.Synth(seed=0xB200, payload_len=1400, plants=1, plant_patterns=strings)
    n = 3_300_000
    nbytes = synth.nbytes(0, n)
    assert nbytes > 2**32 + 2**28
    with kmp.Matcher(0) as m:
        m.set_patterns(strings)
        d_bytes = torch.empty(nbytes + 4096, dtype=torch.uint8, device="cuda:0")
        d_off = torch.empty(n + 1, dtype=torch.int64, device="cuda:0")
        synth.fill_device(m, 0, n, d_bytes.data_ptr(), d_off.data_ptr())
        d_bytes[: n * 1400].view(n, 1400)[::3] = 1  # every third packet without a match
        off = d_off.cpu().numpy()
        k0, k1 = 1, n - 7  # 1400 * 1 = 24 mod 32
        span = (int(off[k0]), int(off[k1]))
        assert span[0] % 32 and span[1] > 2**32
        kn = k1 - k0
        d_counts = torch.zeros(len(strings), dtype=torch.int64, device="cuda:0")
        m.count_device(d_bytes.data_ptr(), d_off.data_ptr() + 8 * k0, kn, d_counts.data_ptr(), span=span)
        torch.cuda.synchronize()
        counts = d_counts.cpu().tolist()
        total = distinct_total(counts, strings)
        d_rec = torch.empty(total * 16, dtype=torch.uint8, device="cuda:0")
        d_n = torch.zeros(1, dtype=torch.int64, device="cuda:0")
        m.find_device(d_bytes.data_ptr(), d_off.data_ptr() + 8 * k0, kn, d_rec.data_ptr(), total, d_n.data_ptr(), span)
        torch.cuda.synchronize()
        assert int(d_n.item()) == total
        want = np.zeros(kn, dtype=bool)
        want[d_rec.cpu().numpy().view(kmp.MATCH_DTYPE)["packet"].astype(np.int64)] = True
        del d_rec
        assert 0 < want.sum() < kn
        d_flags = torch.empty(kn, dtype=torch.uint8, device="cuda:0")
        d_index = torch.empty(kn, dtype=torch.int64, device="cuda:0")
        d_sel = torch.zeros(1, dtype=torch.int64, device="cuda:0")
        d_c2 = torch.zeros(len(strings), dtype=torch.int64, device="cuda:0")
        m.select_device(d_bytes.data_ptr(), d_off.data_ptr() + 8 * k0, kn, d_flags.data_ptr(), span, d_index.data_ptr(),
                        d_sel.data_ptr(), d_c2.data_ptr())
        torch.cuda.synchronize()
        assert np.array_equal(d_flags.cpu().numpy().astype(bool), want)
        assert int(d_sel.item()) == int(want.sum())
        assert np.array_equal(d_index[: int(d_sel.item())].cpu().numpy(), np.flatnonzero(want))
        assert d_c2.cpu().tolist() == counts
        kmp.matcher.check(kmp.lib().kmpb_check_device_errors(m.handle))


def _report_lines(pcap, strings_txt, proto):
    r = subprocess.run([MATCH, pcap, strings_txt, proto], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return [ln for ln in r.stdout.splitlines() if ln.endswith("times!")]


@pytest.mark.gpu
@pytest.mark.parametrize("pcap", PCAPS)
@pytest.mark.parametrize("nocase", [False, True])
def test_kmp_select(strings_txt, tmp_path, pcap, nocase):
    """kmp_match finds on the output every match it finds on the input, and none on the -v output; the two outputs
    partition the accepted frames"""
    path = os.path.join(DATA, pcap + ".pcap")
    proto = "tcp" if pcap == "tcp" else "udp"
    flag = ["-i"] if nocase else []
    outs = {}
    for inv in (False, True):
        out = str(tmp_path / ("out_%d.pcap" % inv))
        r = subprocess.run([SELECT] + flag + (["-v"] if inv else []) + [path, strings_txt, out, proto],
                           capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        m = re.fullmatch(r"(\d+) of (\d+) packets written to (.*)\n", r.stdout)
        assert m and m.group(3) == out, r.stdout
        outs[inv] = (out, int(m.group(1)), int(m.group(2)))
    acc = accepted_frames(path, proto)
    assert outs[False][2] == outs[True][2] == len(acc)
    assert outs[False][1] + outs[True][1] == len(acc)
    want_lines = _report_lines(path, strings_txt, proto)
    assert _report_lines(outs[False][0], strings_txt, proto) == want_lines
    assert _report_lines(outs[True][0], strings_txt, proto) == []
    frames = pcap_frames(path)
    chosen = [pcap_frames(outs[inv][0]) for inv in (False, True)]
    merged, i, j = [], 0, 0
    for f in acc.tolist():  # both outputs are subsequences of the accepted frames that together cover them
        if i < len(chosen[0]) and chosen[0][i] == frames[f]:
            i += 1
        elif j < len(chosen[1]) and chosen[1][j] == frames[f]:
            j += 1
        else:
            raise AssertionError("frame %d is in neither output" % f)
        merged.append(f)
    assert i == len(chosen[0]) and j == len(chosen[1])
