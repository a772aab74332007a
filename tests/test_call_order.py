"""Calls interleaved on one context, and two contexts at once.

The other suites check every count and find form one call at a time, waiting for the device in between.  Here calls
overlap the way a device-resident caller issues them:
  - device-form calls on different streams with no host wait in between (they share slot 0's counters, work counters,
    item table and the sort scratch, so the context runs them in call order on the device);
  - a host-form call, a savefile call, a frame stream or a new pattern set right behind a device-form call still running;
  - a frame stream open while other calls are made: it owns the context's counters and pinned staging slots until it is
    closed, so those calls refuse with KMPB_ESTATE and the stream's counts stay exact;
  - the frame stream's batch edges, against closed-form counts;
  - two contexts driven from two host threads at once (ctypes releases the GIL during a call).
Every answer is exact.  Inputs: A, strings.txt planted into 20 000 packets of 1400 bytes, and B, 12 000 packets of mixed
lengths (also as a savefile and as UDP frames), both checked against the oracle's counts and the reference finder's
records; L, 1 000 000 packets of 1400 bytes generated on the device (1.4 GB, config 3's shape), long enough that the next
call is issued while its kernels run.  L's expected answer is the same call run alone, which must equal the per-pattern
engine's counts and whose records' histogram must equal the counts."""
import itertools
import threading
from types import SimpleNamespace

import numpy as np
import pytest

import bench
import multithreading_string_matching_b200 as kmp
from test_find import RefFinder, assert_invariant

pytestmark = pytest.mark.gpu

ESTATE, ELIMIT = -7, -8
FORMS = ["count_device_span", "count_device", "count_device_span_peers", "find_sorted", "find_unsorted"]
C_NAME = {"count_device_span": "kmpb_count_device_span", "count_device": "kmpb_count_device",
          "count_device_span_peers": "kmpb_count_device_span_peers", "find_sorted": "kmpb_find_device_span",
          "find_unsorted": "kmpb_find_device_span"}


def keys(rec):
    """records -> one uint64 each, in the order of (packet, offset, pattern)"""
    assert len(rec) == 0 or (int(rec["packet"].max()) < 1 << 24 and int(rec["pattern"].max()) < 256)
    return (rec["packet"].astype(np.uint64) << np.uint64(40)) | (rec["offset"].astype(np.uint64) << np.uint64(8)) | \
        rec["pattern"].astype(np.uint64)


def fold(data):
    """ASCII case folding (A-Z to a-z, nothing else) of a uint8 array"""
    out = np.array(data, dtype=np.uint8)
    out[(out >= 0x41) & (out <= 0x5A)] += 0x20
    return out


def udp_frame(payload, proto=17, ihl=5):
    """Ethernet + IPv4 (ihl words) + UDP header + payload"""
    return b"\x02" * 12 + b"\x08\x00" + bytes([0x40 | ihl, 0, 0, 0, 0, 0, 0, 0, 64, proto]) + bytes(10 + 8) + bytes(payload)


def device_copy(data, offsets):
    import torch

    d_bytes = torch.zeros(len(data) + 64, dtype=torch.uint8, device="cuda:0")
    d_bytes[: len(data)] = torch.from_numpy(np.ascontiguousarray(data))
    return d_bytes, torch.from_numpy(offsets.astype(np.int64)).to("cuda:0")


class Call:
    """One device-form call on batch b: its outputs are allocated and cleared up front, so issue() only enqueues."""

    def __init__(self, form, b):
        import torch

        self.form, self.b = form, b
        if form.startswith("find"):
            self.capacity = len(b.keys)
            self.out = torch.full(((self.capacity + 8) * 16,), 0xA5, dtype=torch.uint8, device="cuda:0")
            self.total = torch.full((1,), -1, dtype=torch.int64, device="cuda:0")
        else:
            n_vec = 2 if form == "count_device_span_peers" else 1
            self.vecs = [torch.zeros(len(b.counts), dtype=torch.int64, device="cuda:0") for _ in range(n_vec)]

    def issue(self, m, stream):
        b, s = self.b, None if stream is None else stream.cuda_stream
        ptrs = (b.d_bytes.data_ptr(), b.d_off.data_ptr(), b.n)
        if self.form == "count_device_span":
            m.count_device(*ptrs, self.vecs[0].data_ptr(), span=b.span, stream=s)
        elif self.form == "count_device":
            m.count_device(*ptrs, self.vecs[0].data_ptr(), stream=s)
        elif self.form == "count_device_span_peers":
            m.count_device_into(*ptrs, [v.data_ptr() for v in self.vecs], span=b.span, stream=s)
        else:
            m.find_device(*ptrs, self.out.data_ptr(), self.capacity, self.total.data_ptr(), b.span,
                          sorted=self.form == "find_sorted", stream=s)

    def records(self):
        """(total, records written, canary behind them intact), once the call has finished"""
        raw = self.out.cpu().numpy()
        total = int(self.total.item())
        rec = raw[: 16 * min(max(total, 0), self.capacity)].view(kmp.MATCH_DTYPE)
        return total, rec, bool((raw[16 * self.capacity:] == 0xA5).all())

    def mismatch(self):
        """None if the finished call's answer is b's expected one, else what differs"""
        if not self.form.startswith("find"):
            got = [v.cpu().tolist() for v in self.vecs]
            return None if all(g == self.b.counts for g in got) else "counts differ in %s" % [
                sum(x != y for x, y in zip(g, self.b.counts)) for g in got]
        total, rec, ok = self.records()
        k = keys(rec) if self.form == "find_sorted" else np.sort(keys(rec))
        if total == len(self.b.keys) and ok and np.array_equal(k, self.b.keys):
            return None
        return "total %d (want %d), canary %s, %d records differ" % (
            total, len(self.b.keys), ok, len(np.setxor1d(k, self.b.keys)) if len(k) else len(self.b.keys))


# ---- inputs -------------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def strings(strings_txt):
    return kmp.load_patterns(strings_txt)


@pytest.fixture(scope="module")
def finder(tmp_path_factory):
    return RefFinder(str(tmp_path_factory.mktemp("kmp_find_ref")))


@pytest.fixture(scope="module")
def m(strings):
    with kmp.Matcher(0) as m:
        m.set_patterns(strings)
        yield m


def expected(b, oracle, finder, patterns):
    b.counts = oracle.count_csr(b.data, b.offsets, patterns)
    rec = finder.find_csr(b.data, b.offsets, patterns)
    assert_invariant(b.counts, rec, patterns)
    b.keys = keys(rec)
    assert len(b.keys) > 1000
    return b


@pytest.fixture(scope="module")
def A(oracle, finder, strings):
    data, offsets = kmp.Synth(seed=0xA, payload_len=1400, plants=2, plant_patterns=strings).fill_host(0, 20_000)
    a = expected(SimpleNamespace(data=data, offsets=offsets, n=len(offsets) - 1, span=(0, int(offsets[-1]))),
                 oracle, finder, strings)
    a.d_bytes, a.d_off = device_copy(data, offsets)
    a.other = strings[::5] + [b"zz", b"~~", b"Ab"]  # a second pattern set, and its counts on A
    a.other_counts = oracle.count_csr(data, offsets, a.other)
    return a


@pytest.fixture(scope="module")
def B(oracle, finder, strings, tmp_path_factory):
    data, offsets = kmp.Synth(seed=0xB, len_mode=1, plants=2, plant_patterns=strings).fill_host(0, 12_000)
    b = expected(SimpleNamespace(data=data, offsets=offsets, n=len(offsets) - 1, span=(0, int(offsets[-1]))),
                 oracle, finder, strings)
    assert len(set(np.diff(offsets.astype(np.int64)).tolist())) == 4  # 64, 576, 1400 and 9000 bytes
    b.d_bytes, b.d_off = device_copy(data, offsets)
    b.path = str(tmp_path_factory.mktemp("call_order") / "b.pcap")
    bench.write_pcap(b.path, data, offsets)
    b.frames = [udp_frame(data[int(x):int(y)]) for x, y in zip(offsets[:-1], offsets[1:])]
    return b


@pytest.fixture(scope="module")
def L(m, strings):
    """config 3's shape on the device; its expected answers are each call run alone"""
    import torch

    n = 1_000_000
    synth = kmp.Synth(seed=0xC3, payload_len=1400, plants=2, plant_patterns=strings)
    nbytes = synth.nbytes(0, n)
    d_bytes = torch.empty(nbytes + 4096, dtype=torch.uint8, device="cuda:0")
    d_bytes[nbytes:].zero_()
    d_off = torch.empty(n + 1, dtype=torch.int64, device="cuda:0")
    synth.fill_device(m, 0, n, d_bytes.data_ptr(), d_off.data_ptr())
    torch.cuda.synchronize()
    b = SimpleNamespace(d_bytes=d_bytes, d_off=d_off, n=n, span=(0, nbytes), counts=[0] * len(strings), keys=[])
    alone = Call("count_device_span", b)
    alone.issue(m, None)
    torch.cuda.synchronize()
    b.counts = alone.vecs[0].cpu().tolist()
    m.set_engine("perpat")
    try:
        perpat = Call("count_device_span", b)
        perpat.issue(m, None)
        torch.cuda.synchronize()
    finally:
        m.set_engine("auto")
    assert perpat.vecs[0].cpu().tolist() == b.counts and sum(b.counts) > n
    b.keys = np.zeros(sum(b.counts), dtype=np.uint64)  # at least the number of records: the capacity of the first run
    alone = Call("find_sorted", b)
    alone.issue(m, None)
    torch.cuda.synchronize()
    total, rec, ok = alone.records()
    assert ok and 0 < total <= len(b.keys)
    assert_invariant(b.counts, rec, strings)
    b.keys = keys(rec)
    assert (np.diff(b.keys) > 0).all()
    for form in FORMS:  # and every form alone gives that answer
        alone = Call(form, b)
        alone.issue(m, None)
        torch.cuda.synchronize()
        assert alone.mismatch() is None, form
    return b


# ---- 1. device-form calls on different streams, no host wait in between -------------------------------------------

@pytest.mark.parametrize("engine", ["union", "perpat"])
def test_device_calls_on_two_streams(m, A, L, engine):
    """Every ordered pair (X on L, Y on A) of the device forms, Y on another stream or on the legacy default stream,
    issued back to back; then one synchronise.  Under the per-pattern engine the count forms run it (finding always
    runs the union engine)."""
    import torch

    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    bad = []
    m.set_engine(engine)
    try:
        for x, y in itertools.product(FORMS, FORMS):
            for second in (s2, None):
                cx, cy = Call(x, L), Call(y, A)
                torch.cuda.synchronize()
                cx.issue(m, s1)
                cy.issue(m, second)
                torch.cuda.synchronize()
                for what, c in (("X " + x, cx), ("Y " + y, cy)):
                    err = c.mismatch()
                    if err:
                        bad.append((x, y, "legacy" if second is None else "stream", what, err))
        # three calls that alternate streams
        calls = [(Call("find_unsorted", L), s1), (Call("count_device_span", A), s2), (Call("find_sorted", L), s1),
                 (Call("count_device_span_peers", L), s2), (Call("find_sorted", A), s1)]
        torch.cuda.synchronize()
        for c, s in calls:
            c.issue(m, s)
        torch.cuda.synchronize()
        bad += [("alternating", c.form, c.mismatch()) for c, _ in calls if c.mismatch()]
    finally:
        m.set_engine("auto")
    assert not bad, bad[:6]
    kmp.matcher.check(kmp.lib().kmpb_check_device_errors(m.handle))


# ---- 2. host work right behind a device-form call in flight ---------------------------------------------------------

@pytest.mark.parametrize("work", ["count_host", "find_host", "count_pcap", "find_pcap", "stream", "set_patterns"])
def test_host_work_behind_a_device_call(m, strings, A, B, L, work):
    import torch

    s1 = torch.cuda.Stream()
    bad = []
    for x in FORMS:
        cx = Call(x, L)
        torch.cuda.synchronize()
        cx.issue(m, s1)
        try:
            if work == "count_host":
                ok = m.count_host(A.data, A.offsets) == A.counts
            elif work == "find_host":
                ok = np.array_equal(keys(m.find_host(A.data, A.offsets)), A.keys)
            elif work == "count_pcap":
                ok = m.count_pcap_streamed(B.path) == B.counts
            elif work == "find_pcap":
                rec = m.find_pcap(B.path)[["packet", "offset", "pattern"]].astype(kmp.MATCH_DTYPE)
                ok = np.array_equal(keys(rec), B.keys)
            elif work == "stream":
                with m.stream("udp") as st:
                    for f in B.frames:
                        st.push(f)
                    ok = st.flush() == B.counts and st.packets == B.n
            else:
                m.set_patterns(A.other)
                ok = m.count_host(A.data, A.offsets) == A.other_counts
        finally:
            torch.cuda.synchronize()
            if work == "set_patterns":
                m.set_patterns(strings)
        if not ok:
            bad.append((x, work))
        if cx.mismatch():
            bad.append((x, "the device call", cx.mismatch()))
    assert not bad, bad


# ---- 3. an open frame stream refuses other work and loses nothing ---------------------------------------------------

def test_open_stream_refuses_other_work(m, oracle, strings, A, B):
    import torch

    half = B.n // 2

    def refused(name, call):
        with pytest.raises(kmp.KmpbError) as e:
            call()
        assert e.value.code == ESTATE and "frame stream" in str(e.value) and name in str(e.value), (name, str(e.value))

    with m.stream("udp", batch_bytes=65536) as st:  # ~150 batches of 64 KiB: some are in flight at every call below
        for f in B.frames[:half]:
            st.push(f)
        refused("kmpb_set_patterns", lambda: m.set_patterns(A.other))
        refused("kmpb_set_patterns", lambda: m.set_patterns(strings, nocase=True))
        assert m.patterns == strings and m.nocase == [False] * len(strings)
        refused("kmpb_count_host", lambda: m.count_host(A.data, A.offsets))
        refused("kmpb_find_host", lambda: m.find_host(A.data, A.offsets))
        refused("kmpb_count_pcap", lambda: m.count_pcap_streamed(B.path))
        refused("kmpb_find_pcap", lambda: m.find_pcap(B.path))
        refused("kmpb_reserve_staging", lambda: kmp.matcher.check(kmp.lib().kmpb_reserve_staging(m.handle, 0, 0)))
        refused("kmpb_stream_open", lambda: m.stream("udp"))
        calls = [Call(form, A) for form in FORMS]
        torch.cuda.synchronize()
        for c in calls:
            refused(C_NAME[c.form], lambda: c.issue(m, None))
        st.push(B.frames[half])
        # still allowed: what touches no slot state
        m.set_engine("perpat")  # the later batches run the per-pattern engine
        assert m.prefix(0) == oracle.kmp_prefix(strings[0])
        assert kmp.lib().kmpb_pattern_count(m.handle) == len(strings) and m.launches > 0
        kmp.matcher.check(kmp.lib().kmpb_check_device_errors(m.handle))
        synth = kmp.Synth(seed=3, payload_len=100, plants=1, plant_patterns=strings)
        d_bytes = torch.zeros(synth.nbytes(0, 50) + 64, dtype=torch.uint8, device="cuda:0")
        d_off = torch.zeros(51, dtype=torch.int64, device="cuda:0")
        torch.cuda.synchronize()
        synth.fill_device(m, 0, 50, d_bytes.data_ptr(), d_off.data_ptr())
        hdata, hoff = synth.fill_host(0, 50)
        assert np.array_equal(d_bytes[: len(hdata)].cpu().numpy(), hdata) and d_off.cpu().numpy().tolist() == hoff.tolist()
        for f in B.frames[half + 1:]:
            st.push(f)
        assert st.flush() == B.counts and st.packets == B.n
        assert st.flush() == B.counts
        for c in calls:  # nothing was enqueued
            assert c.form.startswith("find") and int(c.total.item()) == -1 or not c.form.startswith("find") and \
                all(v.abs().sum().item() == 0 for v in c.vecs), c.form
    m.set_engine("auto")
    # closed: every form works again and is exact, and so does a new stream
    assert m.count_host(A.data, A.offsets) == A.counts
    assert np.array_equal(keys(m.find_host(A.data, A.offsets)), A.keys)
    for form in FORMS:
        c = Call(form, A)
        torch.cuda.synchronize()
        c.issue(m, None)
        torch.cuda.synchronize()
        assert c.mismatch() is None, form
    assert m.count_pcap_streamed(B.path) == B.counts
    assert np.array_equal(keys(m.find_pcap(B.path)[["packet", "offset", "pattern"]].astype(kmp.MATCH_DTYPE)), B.keys)
    kmp.matcher.check(kmp.lib().kmpb_reserve_staging(m.handle, 0, 0))
    with m.stream("udp") as st:
        for f in B.frames:
            st.push(f)
        assert st.flush() == B.counts
    m.set_patterns(A.other)
    assert m.count_host(A.data, A.offsets) == A.other_counts
    m.set_patterns(strings)


# ---- 4. the frame stream's batch edges, against closed-form counts --------------------------------------------------

EDGE_PATTERNS = [b"ab", b"a", b"b", b"ba", b"abab"]


def ab_counts(k):
    """EDGE_PATTERNS in one payload of "ab" * k"""
    return [k, k, k, k - 1, k - 1] if k else [0] * 5


def test_stream_batch_edges():
    with kmp.Matcher(0) as e:
        e.set_patterns(EDGE_PATTERNS)
        with e.stream("udp", batch_bytes=65536) as st:
            assert st.flush() == [0] * 5 and st.flush() == [0] * 5 and st.packets == 0  # nothing pushed
            st.push(udp_frame(b"ab" * 32768))  # exactly batch_bytes
            assert st.flush() == ab_counts(32768) and st.flush() == ab_counts(32768)
            st.push(udp_frame(b"ab" * 32768))
            st.push(udp_frame(b"ab"))  # the full batch goes first
            with pytest.raises(kmp.KmpbError) as err:
                st.push(udp_frame(b"a" * 65537))  # batch_bytes + 1
            assert err.value.code == ELIMIT and "does not fit" in str(err.value)
            for refused in (udp_frame(b"abab" * 8, proto=6),  # TCP in a UDP stream
                            udp_frame(b"abab", ihl=15)[:60],  # an IP header longer than the frame
                            udp_frame(b"")[:40], b"", b"\x02" * 13):  # shorter than the headers
                st.push(refused)
            st.push(udp_frame(b"ab"))
            want = [2 * x + 2 * y for x, y in zip(ab_counts(32768), ab_counts(1))]
            assert st.packets == 4
            assert st.flush() == want and st.flush() == want
        # 2^20 + 3 two-byte payloads: batches end at the per-batch packet limit (2^20) before they fill 4 MiB
        n = (1 << 20) + 3
        with e.stream("udp", batch_bytes=4 << 20) as st:
            push, h, f = kmp.lib().kmpb_stream_push, st._s, udp_frame(b"ab")
            failed = sum(1 for _ in range(n) if push(h, f, len(f)))
            assert failed == 0 and st.packets == n
            assert st.flush() == [n, n, n, 0, 0]  # no match across two packets, none lost at the batch's end
            st.push(udp_frame(b"ba"))
            assert st.flush() == [n, n + 1, n + 1, 1, 0]


# ---- 5. two contexts, two host threads ------------------------------------------------------------------------------

def test_two_contexts_two_threads(oracle, finder, strings, A, B):
    """Each context has its own pattern set (one of them all nocase) and its own batch; their calls overlap."""
    import torch

    nc = [p.upper() if i % 2 else p.swapcase() for i, p in enumerate(strings)] + [b"HtTp", b"UDP"]
    folded = fold(B.data)
    jobs = [SimpleNamespace(patterns=strings, nocase=False, b=A, counts=A.counts, keys=A.keys),
            SimpleNamespace(patterns=nc, nocase=True, b=B, counts=oracle.count_csr(folded, B.offsets, [p.lower() for p in nc]),
                            keys=keys(finder.find_csr(folded, B.offsets, [p.lower() for p in nc])))]
    assert jobs[1].counts != oracle.count_csr(B.data, B.offsets, nc)
    errors = []
    start = threading.Barrier(len(jobs))

    def run(job):
        try:
            stream = torch.cuda.Stream()
            d_counts = torch.zeros(len(job.patterns), dtype=torch.int64, device="cuda:0")
            torch.cuda.synchronize()
            start.wait()
            for r in range(4):
                assert job.m.count_host(job.b.data, job.b.offsets) == job.counts, ("count_host", r)
                assert np.array_equal(keys(job.m.find_host(job.b.data, job.b.offsets)), job.keys), ("find_host", r)
                with torch.cuda.stream(stream):
                    d_counts.zero_()
                    job.m.count_device(job.b.d_bytes.data_ptr(), job.b.d_off.data_ptr(), job.b.n, d_counts.data_ptr(),
                                       stream=stream.cuda_stream)
                stream.synchronize()
                assert d_counts.cpu().tolist() == job.counts, ("count_device", r)
        except BaseException as exc:  # noqa: B902 -- reported by the main thread
            errors.append((job.nocase, repr(exc)[:500]))

    for job in jobs:
        job.m = kmp.Matcher(0)
        job.m.set_patterns(job.patterns, nocase=job.nocase)
    try:
        threads = [threading.Thread(target=run, args=(job,)) for job in jobs]
        for t in threads:
            t.start()
        for t in threads:
            t.join()
    finally:
        for job in jobs:
            job.m.close()
    assert not errors, errors
