// api.cu -- the C ABI of include/kmpb200.h: context, pattern upload, the two count entry points.
#include <algorithm>
#include <new>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>
#include <vector>

#include "kmpb_device.cuh"

namespace {

int use_device(const kmpb_ctx *ctx)
{
    KMPB_CUDA(cudaSetDevice(ctx->device));
    return KMPB_OK;
}

bool device_is_sm100(int device)
{
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return false;
    return prop.major == 10; // the library carries sm_100a code only
}

// counts[i] (+)= sum over slots of uniq_counts[slot][pat_to_uniq[i]].  accumulate: 0 = overwrite, 1 = add (the vector
// is this caller's alone), 2 = add with system-scope atomics (the vector may be a peer GPU's, mapped over NVLink, and
// other ranks may be adding to it at the same time)
__global__ void kmpb_expand_counts_kernel(const unsigned long long *__restrict__ uniq_counts, uint32_t n_uniq,
                                          int n_slots, const uint32_t *__restrict__ pat_to_uniq, uint32_t n_pat,
                                          unsigned long long *__restrict__ counts, int accumulate)
{
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_pat) return;
    const uint32_t u = pat_to_uniq[i];
    unsigned long long v = 0ull;
    for (int s = 0; s < n_slots; s++) v += uniq_counts[(size_t)s * n_uniq + u];
    if (accumulate == 2) {
        if (v) atomicAdd_system(counts + i, v);
    } else {
        counts[i] = (accumulate ? counts[i] : 0ull) + v;
    }
}

int run_engine(kmpb_ctx *ctx, const kmpb_batch &b, int slot, cudaStream_t stream)
{
    uint64_t *acc = ctx->d_uniq_counts + (size_t)slot * ctx->host.n_uniq;
    if (ctx->engine == KMPB_ENGINE_PERPAT) return kmpb_launch_perpat(ctx, b, acc, stream);
    return kmpb_launch_union(ctx, b, slot, acc, stream);
}

// everything a chunked form needs for chunks of up to max_bytes / max_pkts: the device staging slots (zero-filled when
// new), their pinned twins when the chunks are packed on the host first, the union engine's scratch
int reserve(kmpb_ctx *ctx, uint64_t max_bytes, uint64_t max_pkts, bool pinned)
{
    for (int i = 0; i < KMPB_COPY_STREAMS; i++) {
        int rc;
        if ((rc = ctx->d_stage_bytes[i].reserve(max_bytes + 1024, true)) || (rc = ctx->d_stage_off[i].reserve(max_pkts + 1)) ||
            (pinned && ((rc = ctx->h_stage_bytes[i].reserve(max_bytes + 1024)) || (rc = ctx->h_stage_off[i].reserve(max_pkts + 1)))))
            return rc;
    }
    return kmpb_union_scratch(ctx, max_bytes);
}

// The host may write a slot's pinned buffers again once their last copy to the device has left them.  (An event never
// recorded, or recorded by an earlier call that has finished, is complete: the wait returns at once.)
int wait_pinned(kmpb_ctx *ctx, int slot)
{
    KMPB_CUDA(cudaEventSynchronize(ctx->ev_h2d[slot]));
    return KMPB_OK;
}

// the n packets (nbytes of payload) packed into the slot's pinned buffers to its device twin, on the slot's stream
int submit_pinned(kmpb_ctx *ctx, int slot, uint64_t n, uint64_t nbytes, kmpb_batch &b)
{
    cudaStream_t s = ctx->copy_stream[slot];
    uint8_t *h_bytes = ctx->h_stage_bytes[slot].p, *d_bytes = ctx->d_stage_bytes[slot].p;
    uint64_t *d_off = ctx->d_stage_off[slot].p;
    memset(h_bytes + nbytes, 0, 64);
    KMPB_CUDA(cudaMemcpyAsync(d_bytes, h_bytes, nbytes + 64, cudaMemcpyHostToDevice, s));
    KMPB_CUDA(cudaMemcpyAsync(d_off, ctx->h_stage_off[slot].p, (n + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, s));
    KMPB_CUDA(cudaEventRecord(ctx->ev_h2d[slot], s));
    b = kmpb_batch{d_bytes, 0, d_off, n, 0, nbytes};
    return KMPB_OK;
}

// sums the per-slot accumulators into file order, copies them out and reports device-side error flags
int finish_chunked(kmpb_ctx *ctx, int n_slots, uint64_t *counts_out)
{
    const uint32_t n_pat = ctx->host.n_pat, nu = ctx->host.n_uniq;
    for (int s = 0; s < n_slots; s++) {
        KMPB_CUDA(cudaEventRecord(ctx->ev[3], ctx->copy_stream[s]));
        KMPB_CUDA(cudaStreamWaitEvent(ctx->stream, ctx->ev[3], 0));
    }
    kmpb_expand_counts_kernel<<<(n_pat + 255) / 256, 256, 0, ctx->stream>>>(
        (const unsigned long long *)ctx->d_uniq_counts, nu, KMPB_COPY_STREAMS, ctx->dev.pat_to_uniq, n_pat,
        (unsigned long long *)ctx->d_counts, 0);
    ctx->launches++;
    KMPB_CUDA(cudaGetLastError());
    KMPB_CUDA(cudaMemcpyAsync(counts_out, ctx->d_counts, (size_t)n_pat * sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->stream));
    KMPB_CUDA(cudaEventRecord(ctx->ev[1], ctx->stream));
    KMPB_CUDA(cudaStreamSynchronize(ctx->stream));
    float ms = 0;
    KMPB_CUDA(cudaEventElapsedTime(&ms, ctx->ev[0], ctx->ev[1]));
    ctx->last_ms[0] = ms;
    ctx->last_ms[1] = 0;
    return KMPB_OK; // (no device-side flags to read: check_offsets, check_pcap_lengths or kmpb_stream_push checked
                    // every packet's size before anything ran)
}

// bytes per chunk of the chunked forms: 64 MiB, or KMPB_CHUNK_MB
uint64_t chunk_bytes_setting()
{
    uint64_t chunk_bytes = 64ull << 20;
    if (const char *env = getenv("KMPB_CHUNK_MB")) {
        long mb = atol(env);
        if (mb > 0) chunk_bytes = (uint64_t)mb << 20;
    }
    return chunk_bytes;
}

// every offset, not a sample: a decreasing pair anywhere would size a copy wrongly, a packet of KMPB_PACKET_LIMIT bytes
// or more would be skipped by the union engine (one pass over 8 bytes per packet, all host threads; nothing next to
// copying the packets themselves)
int check_offsets(const uint64_t *offsets, uint64_t n_packets)
{
    int64_t bad = -1, big = -1;
#pragma omp parallel for schedule(static) reduction(max : bad, big)
    for (int64_t k = 0; k < (int64_t)n_packets; k++) {
        if (offsets[k + 1] < offsets[k]) bad = k > bad ? k : bad;
        else if (offsets[k + 1] - offsets[k] >= KMPB_PACKET_LIMIT) big = k > big ? k : big;
    }
    if (bad >= 0) return kmpb_fail(KMPB_EINVAL, "offsets decrease at packet %lld", (long long)bad);
    if (big >= 0)
        return kmpb_fail(KMPB_ELIMIT, "packet %lld is %llu bytes long; packets must be shorter than %llu (2 GiB - 1 MiB)",
                         (long long)big, (unsigned long long)(offsets[big + 1] - offsets[big]), KMPB_PACKET_LIMIT);
    return KMPB_OK;
}

// the savefile forms' twin of check_offsets' size check, over accepted packets [first, first+count)
int check_pcap_lengths(const kmpb_pcap *pc, uint64_t first, uint64_t count)
{
    const uint64_t k = kmpb_pcap_first_long(pc, first, count, KMPB_PACKET_LIMIT);
    if (k == first + count) return KMPB_OK;
    return kmpb_fail(KMPB_ELIMIT, "packet %llu has a payload of %llu bytes (2 GiB - 1 MiB) or more; packets must be shorter",
                     (unsigned long long)k, KMPB_PACKET_LIMIT);
}

// Chunk plan of the chunked forms: packets [k0, k1) of every chunk, whole packets of ~chunk_bytes each (a packet larger
// than a chunk still travels whole), and the largest chunk's bytes and packets, which the staging slots must hold.
// Chunk c goes to stream slot c % KMPB_COPY_STREAMS; k0 is also the packet index the find records of the chunk start at.
struct chunk { uint64_t k0, k1; };
struct chunk_plan {
    std::vector<chunk> chunks;
    uint64_t max_bytes = 0, max_pkts = 0;
    void add(uint64_t k0, uint64_t k1, uint64_t bytes)
    {
        chunks.push_back({k0, k1});
        max_bytes = std::max(max_bytes, bytes);
        max_pkts = std::max(max_pkts, k1 - k0);
    }
    int slots() const { return (int)std::min<size_t>(KMPB_COPY_STREAMS, chunks.size()); }
};

// a host batch; a chunk's bytes count from its 512-byte aligned base
chunk_plan plan_host(const uint64_t *offsets, uint64_t n_packets, uint64_t chunk_bytes)
{
    chunk_plan plan;
    for (uint64_t k0 = 0; k0 < n_packets;) {
        const uint64_t want = offsets[k0] + chunk_bytes;
        uint64_t k1 = (uint64_t)(std::lower_bound(offsets + k0 + 1, offsets + n_packets, want) - offsets);
        if (k1 > n_packets) k1 = n_packets;
        k1 = std::min<uint64_t>(k1, k0 + ((1ull << 31) - 2));
        plan.add(k0, k1, offsets[k1] - (offsets[k0] & ~511ull));
        k0 = k1;
    }
    return plan;
}

// accepted packets [first, last) of a savefile, at most 2^22 packets a chunk
chunk_plan plan_pcap(const kmpb_pcap *pc, uint64_t first, uint64_t last, uint64_t chunk_bytes)
{
    chunk_plan plan;
    for (uint64_t k0 = first; k0 < last;) {
        uint64_t bytes = 0;
        const uint64_t k1 = kmpb_pcap_chunk_end(pc, k0, last, chunk_bytes, 1ull << 22, &bytes);
        plan.add(k0, k1, bytes);
        k0 = k1;
    }
    return plan;
}

double now_s() { timespec ts; clock_gettime(CLOCK_MONOTONIC, &ts); return ts.tv_sec + 1e-9 * ts.tv_nsec; }

int init_context(kmpb_ctx *ctx)
{
    const int device = ctx->device;
    KMPB_CUDA(cudaSetDevice(device));
    int v = 0;
    KMPB_CUDA(cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, device));
    ctx->sm_count = v;
    KMPB_CUDA(cudaDeviceGetAttribute(&v, cudaDevAttrMaxSharedMemoryPerBlockOptin, device));
    ctx->smem_optin = (size_t)v;
    KMPB_CUDA(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
    for (auto &s : ctx->copy_stream) KMPB_CUDA(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
    for (auto &ev : ctx->ev) KMPB_CUDA(cudaEventCreate(&ev));
    for (auto &ev : ctx->ev_kernel) KMPB_CUDA(cudaEventCreate(&ev));
    for (auto &ev : ctx->ev_h2d) KMPB_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    KMPB_CUDA(cudaEventCreateWithFlags(&ctx->ev_dev, cudaEventDisableTiming));
    return KMPB_OK;
}

// An open frame stream owns the context until kmpb_stream_close: its batches accumulate in the per-slot counters and
// its partly filled batch sits in a pinned staging slot, both of which every count and find form, kmpb_set_patterns
// and kmpb_reserve_staging reuse.  Those calls refuse while a stream is open (they call this first).
int no_open_stream(const kmpb_ctx *ctx, const char *call)
{
    if (ctx->open_streams == 0) return KMPB_OK;
    return kmpb_fail(KMPB_ESTATE, "%s while a frame stream (kmpb_stream_open) is open on this context: close the stream "
                     "first, or use a second context", call);
}

// Device-form calls of one context run in call order, whatever streams they are issued on: each makes its stream wait
// for ev_dev, which the previous one recorded after its last enqueued work, and records ev_dev after its own.  The host
// forms and kmpb_stream_open make the streams they start on wait for it as well, so they run after every device-form
// call issued before them.  Nothing here waits on the host.  (An event never recorded is complete.)
int after_device_calls(kmpb_ctx *ctx, cudaStream_t stream)
{
    KMPB_CUDA(cudaStreamWaitEvent(stream, ctx->ev_dev, 0));
    return KMPB_OK;
}

template <class Enqueue>
int device_ordered(kmpb_ctx *ctx, cudaStream_t stream, Enqueue &&enqueue)
{
    int rc = after_device_calls(ctx, stream);
    if (rc) return rc;
    rc = enqueue();
    const cudaError_t e = cudaEventRecord(ctx->ev_dev, stream); // also after a failure: whatever was enqueued is covered
    if (rc) return rc;
    KMPB_CUDA(e);
    return KMPB_OK;
}

// every copy stream idle again: an error return must not leave copies or kernels of the call in flight
void quiesce(kmpb_ctx *ctx)
{
    for (auto &s : ctx->copy_stream)
        if (s) cudaStreamSynchronize(s);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    cudaGetLastError();
}

// The start of a chunked call or a frame stream: after every device-form call issued before it, ev[0] recorded (where
// the interval of kmpb_last_timing begins), the slots' distinct-pattern counters zeroed, and the copy streams of the
// first n_slots slots behind all of that.
int start_chunks(kmpb_ctx *ctx, int n_slots)
{
    int rc = after_device_calls(ctx, ctx->stream);
    if (rc) return rc;
    KMPB_CUDA(cudaEventRecord(ctx->ev[0], ctx->stream));
    KMPB_CUDA(cudaMemsetAsync(ctx->d_uniq_counts, 0, (size_t)KMPB_COPY_STREAMS * ctx->host.n_uniq * sizeof(uint64_t), ctx->stream));
    KMPB_CUDA(cudaEventRecord(ctx->ev[2], ctx->stream));
    for (int s = 0; s < n_slots; s++) KMPB_CUDA(cudaStreamWaitEvent(ctx->copy_stream[s], ctx->ev[2], 0));
    return KMPB_OK;
}

// The chunk pipeline of every host and savefile form.  Chunk c goes to stream slot c % KMPB_COPY_STREAMS: once the
// slot's previous chunk, c - KMPB_COPY_STREAMS, is retired, the input stages chunk c into the slot's staging buffers
// and enqueue(batch, slot) puts the operation's work on the slot's stream.  So the copies and kernels of the chunks in
// between keep the device busy while the host retires a chunk.  The last iterations retire the last chunks.  An
// operation supplies enqueue and retire(chunk, slot, batch); nothing of the call is left in flight when it returns an
// error.
template <class Input, class Enqueue, class Retire>
int run_chunks(kmpb_ctx *ctx, Input &in, Enqueue &&enqueue, Retire &&retire)
{
    const std::vector<chunk> &chunks = in.plan.chunks;
    kmpb_batch batch[KMPB_COPY_STREAMS] = {};
    int rc = start_chunks(ctx, in.plan.slots());
    for (size_t c = 0; c < chunks.size() + KMPB_COPY_STREAMS && !rc; c++) {
        const int slot = (int)(c % KMPB_COPY_STREAMS);
        if (c >= (size_t)KMPB_COPY_STREAMS && (rc = retire(chunks[c - KMPB_COPY_STREAMS], slot, batch[slot]))) break;
        if (c < chunks.size() && !(rc = in.stage(ctx, chunks[c], slot, batch[slot]))) rc = enqueue(batch[slot], slot);
    }
    if (rc) quiesce(ctx);
    return rc;
}

// The two inputs of the chunked forms.  in_range() checks the packet range; prepare() checks the input, selects the
// device, plans the chunks (none for an empty input: the call has nothing more to do) and reserves the staging slots;
// stage() puts a chunk into its slot's device buffers, copies on the slot's stream.  k_base is the packet index of the
// input's first packet.
//
// A host CSR batch: a chunk is copied from the caller's memory, from its 512-byte aligned base (the MPI variant's
// Scatterv, done by the copy engines instead of the network: mpi_dumping.c:161).
struct host_input {
    const uint8_t *bytes;
    const uint64_t *offsets;
    uint64_t n; // packets
    uint64_t k_base = 0;
    chunk_plan plan;

    int in_range() const { return KMPB_OK; }

    int prepare(kmpb_ctx *ctx)
    {
        if (n == 0) return KMPB_OK;
        if (bytes == nullptr || offsets == nullptr) return kmpb_fail(KMPB_EINVAL, "NULL batch pointer");
        int rc = check_offsets(offsets, n);
        if (rc || (rc = use_device(ctx))) return rc;
        plan = plan_host(offsets, n, chunk_bytes_setting());
        return reserve(ctx, plan.max_bytes, plan.max_pkts, false);
    }

    int stage(kmpb_ctx *ctx, const chunk &ch, int slot, kmpb_batch &b)
    {
        cudaStream_t s = ctx->copy_stream[slot];
        const uint64_t k0 = ch.k0, k1 = ch.k1, base = offsets[k0] & ~511ull;
        uint8_t *d_bytes = ctx->d_stage_bytes[slot].p;
        uint64_t *d_off = ctx->d_stage_off[slot].p;
        KMPB_CUDA(cudaMemcpyAsync(d_bytes, bytes + base, offsets[k1] - base, cudaMemcpyHostToDevice, s));
        KMPB_CUDA(cudaMemcpyAsync(d_off, offsets + k0, (k1 - k0 + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, s));
        b = kmpb_batch{d_bytes, base, d_off, k1 - k0, offsets[k0], offsets[k1]};
        return KMPB_OK;
    }

    void report(const char *) const {} // (no waiting or packing to report)
};

// Accepted packets [k_base, k_base + n) of a savefile: a chunk is packed into the slot's pinned buffers (all host
// threads), then copied over while the next chunk is packed -- the producer/consumer shape of openmp_task.c:113-178
// with the GPU as the consumer.  t[0] and t[1] add up the seconds spent waiting for the slot and packing since t0.
struct pcap_input {
    const kmpb_pcap *pc;
    uint64_t k_base, n;
    chunk_plan plan;
    double t0 = 0, t[2] = {0, 0};

    int in_range() const
    {
        const uint64_t total = kmpb_pcap_packets(pc);
        if (k_base > total || n > total - k_base) return kmpb_fail(KMPB_EINVAL, "packet range outside the file");
        return KMPB_OK;
    }

    int prepare(kmpb_ctx *ctx)
    {
        int rc = in_range();
        if (rc || n == 0) return rc;
        if ((rc = check_pcap_lengths(pc, k_base, n)) || (rc = use_device(ctx))) return rc;
        plan = plan_pcap(pc, k_base, k_base + n, chunk_bytes_setting());
        rc = reserve(ctx, plan.max_bytes, plan.max_pkts, true);
        t0 = now_s();
        return rc;
    }

    int stage(kmpb_ctx *ctx, const chunk &ch, int slot, kmpb_batch &b)
    {
        const uint64_t k = ch.k1 - ch.k0;
        const double s0 = now_s();
        const int rc = wait_pinned(ctx, slot);
        if (rc) return rc;
        const double s1 = now_s();
        kmpb_pcap_pack(pc, ch.k0, k, ctx->h_stage_bytes[slot].p, ctx->h_stage_off[slot].p);
        t[0] += s1 - s0;
        t[1] += now_s() - s1;
        return submit_pinned(ctx, slot, k, ctx->h_stage_off[slot].p[k], b);
    }

    void report(const char *call) const
    {
        fprintf(stderr, "%s: %llu chunks; waiting for a free slot %.3f s, packing %.3f s, issuing copies and kernels %.3f s\n",
                call, (unsigned long long)plan.chunks.size(), t[0], t[1], now_s() - t0 - t[0] - t[1]);
    }
};

// Counting: the count engine adds every chunk into its slot's accumulators, finish_chunked sums them.
template <class Input>
int count_chunked(kmpb_ctx *ctx, Input &in, uint64_t *counts_out, const char *call)
{
    if (ctx == nullptr) return kmpb_fail(KMPB_EINVAL, "NULL context");
    if (int rc = no_open_stream(ctx, call)) return rc;
    if (!ctx->have_tables) return kmpb_fail(KMPB_ESTATE, "count before kmpb_set_patterns");
    const uint32_t n_pat = ctx->host.n_pat;
    if (n_pat == 0) return KMPB_OK;
    if (counts_out == nullptr) return kmpb_fail(KMPB_EINVAL, "NULL counts_out");
    memset(counts_out, 0, (size_t)n_pat * sizeof(uint64_t));
    int rc = in.prepare(ctx);
    if (rc || in.plan.chunks.empty()) return rc;
    auto enqueue = [&](const kmpb_batch &b, int slot) { return run_engine(ctx, b, slot, ctx->copy_stream[slot]); };
    auto retire = [](const chunk &, int, const kmpb_batch &) { return KMPB_OK; };
    if ((rc = run_chunks(ctx, in, enqueue, retire))) return rc;
    if (getenv("KMPB_STATS")) in.report(call);
    return finish_chunked(ctx, in.plan.slots(), counts_out);
}

// the record buffer of a stream slot of the chunked find forms, at least `records` long (grown by an eighth more)
int ensure_find_rec(kmpb_ctx *ctx, int slot, uint64_t records)
{
    kmpb_scratch<kmpb_match> &rec = ctx->d_find_rec[slot];
    if (rec.p && records <= rec.cap) return KMPB_OK;
    return rec.reserve(records + records / 8 + 1024);
}

// the argument checks every find form starts with
int find_args(kmpb_ctx *ctx, const void *out, uint64_t capacity, const void *n_found, const char *call)
{
    if (ctx == nullptr || n_found == nullptr || (out == nullptr && capacity)) return kmpb_fail(KMPB_EINVAL, "NULL argument");
    if (int rc = no_open_stream(ctx, call)) return rc;
    if (!ctx->have_tables) return kmpb_fail(KMPB_ESTATE, "find before kmpb_set_patterns");
    return KMPB_OK;
}

// Finding: the find kernel writes a chunk's records into its slot's buffer, sized for one record per 256 bytes of the
// largest chunk.  Retiring a chunk reads its match count, then sorts its records and copies them out behind the
// previous chunk's.  A chunk whose records overflowed the slot's buffer is matched again, from the copy still on the
// device, into a buffer of the exact size; once `capacity` records are out, later chunks are only counted.
template <class Input>
int find_chunked(kmpb_ctx *ctx, Input &in, kmpb_match *out, uint64_t capacity, uint64_t *n_found, const char *call)
{
    int rc = find_args(ctx, out, capacity, n_found, call);
    if (rc) return rc;
    *n_found = 0;
    if (ctx->host.n_pat == 0) return KMPB_OK;
    if ((rc = in.prepare(ctx)) || in.plan.chunks.empty() || (rc = ctx->d_find_found.reserve(KMPB_COPY_STREAMS))) return rc;
    for (int s = 0; s < in.plan.slots(); s++)
        if ((rc = ensure_find_rec(ctx, s, in.plan.max_bytes / 256))) return rc;
    uint64_t total = 0, written = 0;
    auto enqueue = [&](const kmpb_batch &b, int slot) {
        return kmpb_find_match(ctx, b, slot, ctx->d_find_rec[slot].p, ctx->d_find_rec[slot].cap, ctx->d_find_found.p + slot,
                               ctx->copy_stream[slot]);
    };
    auto retire = [&](const chunk &ch, int slot, const kmpb_batch &b) -> int {
        cudaStream_t s = ctx->copy_stream[slot];
        unsigned long long *found = ctx->d_find_found.p + slot;
        unsigned long long n = 0;
        KMPB_CUDA(cudaMemcpyAsync(&n, found, sizeof n, cudaMemcpyDeviceToHost, s));
        KMPB_CUDA(cudaStreamSynchronize(s));
        const uint64_t take = std::min<uint64_t>(n, capacity - written);
        if (take) {
            int rc2;
            if (n > ctx->d_find_rec[slot].cap &&
                ((rc2 = ensure_find_rec(ctx, slot, n)) || (rc2 = kmpb_find_match(ctx, b, slot, ctx->d_find_rec[slot].p, n, found, s))))
                return rc2;
            if ((rc2 = kmpb_find_finish(ctx, b, ch.k0, ctx->d_find_rec[slot].p, n, found, true, s))) return rc2;
            KMPB_CUDA(cudaMemcpyAsync(out + written, ctx->d_find_rec[slot].p, take * sizeof(kmpb_match), cudaMemcpyDeviceToHost, s));
            KMPB_CUDA(cudaStreamSynchronize(s));
        }
        total += n;
        written += take;
        return KMPB_OK;
    };
    if ((rc = run_chunks(ctx, in, enqueue, retire))) return rc;
    *n_found = total;
    return KMPB_OK; // (as in finish_chunked: the input's checks covered every packet's size)
}

// the bitmaps and verdict buffers of the chunked select forms: those of the slots the plan uses, for chunks of up to
// max_bytes / max_pkts (a single chunk of one packet close to 2 GiB takes one 256 MiB bitmap, not four)
int reserve_select(kmpb_ctx *ctx, const chunk_plan &plan)
{
    for (int s = 0; s < plan.slots(); s++) {
        int rc;
        if ((rc = kmpb_ensure_mark(ctx, s, plan.max_bytes / 32 + 8, ctx->copy_stream[s])) ||
            (rc = ctx->d_sel_flags[s].reserve(plan.max_pkts)) || (rc = ctx->h_sel_flags[s].reserve(plan.max_pkts)))
            return rc;
    }
    return KMPB_OK;
}

// the argument checks every select form starts with
int select_args(kmpb_ctx *ctx, const void *flags_out, uint64_t n_packets, const char *call)
{
    if (ctx == nullptr || (flags_out == nullptr && n_packets)) return kmpb_fail(KMPB_EINVAL, "NULL argument");
    if (int rc = no_open_stream(ctx, call)) return rc;
    if (!ctx->have_tables) return kmpb_fail(KMPB_ESTATE, "select before kmpb_set_patterns");
    return KMPB_OK;
}

// Selecting: every chunk's mark kernel and verdict pass run into the slot's bitmap and verdicts, which are copied to the
// slot's pinned twin; retiring a chunk copies its verdicts out (flags_out[k - k_base] is packet k's) and counts its
// selected packets.  The counts go to the slots' accumulators as in counting, summed only when counts_out is given.
// The packet range is checked before any output is written.
template <class Input>
int select_chunked(kmpb_ctx *ctx, Input &in, uint8_t *flags_out, uint64_t *n_selected, uint64_t *counts_out, const char *call)
{
    int rc = select_args(ctx, flags_out, in.n, call);
    if (rc || (rc = in.in_range())) return rc;
    const uint32_t n_pat = ctx->host.n_pat;
    if (n_selected) *n_selected = 0;
    if (counts_out) memset(counts_out, 0, (size_t)n_pat * sizeof(uint64_t));
    if (in.n) memset(flags_out, 0, in.n);
    if (n_pat == 0) return KMPB_OK;
    if ((rc = in.prepare(ctx)) || in.plan.chunks.empty() || (rc = reserve_select(ctx, in.plan))) return rc;
    uint64_t selected = 0;
    auto enqueue = [&](const kmpb_batch &b, int slot) -> int {
        cudaStream_t s = ctx->copy_stream[slot];
        if (int rc2 = kmpb_select_match(ctx, b, slot, ctx->d_sel_flags[slot].p, s)) return rc2;
        const cudaError_t e = cudaMemcpyAsync(ctx->h_sel_flags[slot].p, ctx->d_sel_flags[slot].p, b.n_packets, cudaMemcpyDeviceToHost, s);
        return e == cudaSuccess ? KMPB_OK : kmpb_fail(KMPB_ECUDA, "verdict copy failed: %s", cudaGetErrorString(e));
    };
    auto retire = [&](const chunk &ch, int slot, const kmpb_batch &) -> int {
        KMPB_CUDA(cudaStreamSynchronize(ctx->copy_stream[slot]));
        const uint8_t *f = ctx->h_sel_flags[slot].p;
        for (uint64_t j = 0; j < ch.k1 - ch.k0; j++) selected += f[j];
        memcpy(flags_out + (ch.k0 - in.k_base), f, ch.k1 - ch.k0);
        return KMPB_OK;
    };
    if ((rc = run_chunks(ctx, in, enqueue, retire))) return rc;
    if (n_selected) *n_selected = selected;
    return counts_out ? finish_chunked(ctx, in.plan.slots(), counts_out) : KMPB_OK;
}

} // namespace

extern "C" {

int kmpb_device_count(void)
{
    int n = 0, usable = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    for (int d = 0; d < n; d++) usable += device_is_sm100(d) ? 1 : 0;
    return usable;
}

int kmpb_device_ordinal(int index)
{
    int n = 0;
    if (index < 0 || cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return -1; }
    for (int d = 0; d < n; d++)
        if (device_is_sm100(d) && index-- == 0) return d;
    return -1;
}

int kmpb_check_device_errors(kmpb_ctx *ctx)
{
    if (ctx == nullptr) return kmpb_fail(KMPB_EINVAL, "NULL context");
    int rc = use_device(ctx);
    if (rc) return rc;
    KMPB_CUDA(cudaDeviceSynchronize());
    if (ctx->d_work.p == nullptr) return KMPB_OK;
    // the union engine's error flags, word 1 of every slot's work counters: set by its kernels, cleared only here
    uint32_t work[KMPB_COPY_STREAMS * 4];
    KMPB_CUDA(cudaMemcpy(work, ctx->d_work.p, sizeof work, cudaMemcpyDeviceToHost));
    bool flagged = false;
    for (int s = 0; s < KMPB_COPY_STREAMS; s++) flagged |= work[s * 4 + 1] != 0;
    if (!flagged) return KMPB_OK;
    KMPB_CUDA(cudaMemset(ctx->d_work.p, 0, sizeof work));
    return kmpb_fail(KMPB_ELIMIT, "a device-form batch held a packet of %llu bytes (2 GiB - 1 MiB) or more: its results are "
                     "unspecified", KMPB_PACKET_LIMIT);
}

int kmpb_create(kmpb_ctx **out, int device)
{
    if (out == nullptr) return kmpb_fail(KMPB_EINVAL, "kmpb_create: NULL out pointer");
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
        cudaGetLastError();
        return kmpb_fail(KMPB_ENODEVICE, "no CUDA device (%s); libkmpb200 has no CPU path",
                         e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
    }
    if (device < 0 || device >= n) return kmpb_fail(KMPB_EINVAL, "device %d out of range (0..%d)", device, n - 1);
    if (!device_is_sm100(device))
        return kmpb_fail(KMPB_ENODEVICE, "device %d is not compute capability 10.x; libkmpb200 carries sm_100a code only", device);
    kmpb_ctx *ctx = new (std::nothrow) kmpb_ctx();
    if (ctx == nullptr) return kmpb_fail(KMPB_ENOMEM, "out of memory");
    ctx->device = device;
    const int rc = init_context(ctx);
    if (rc != KMPB_OK) { // whatever was created so far goes away again; *out stays NULL
        kmpb_destroy(ctx);
        return rc;
    }
    *out = ctx;
    return KMPB_OK;
}

void kmpb_destroy(kmpb_ctx *ctx)
{
    if (ctx == nullptr) return;
    cudaSetDevice(ctx->device);
    cudaDeviceSynchronize();
    kmpb_release_tables(ctx);
    ctx->d_work.release();
    ctx->d_items.release();
    ctx->d_find_found.release();
    ctx->d_sort_keys[0].release();
    ctx->d_sort_keys[1].release();
    ctx->d_sort_temp.release();
    ctx->d_select_temp.release();
    for (int i = 0; i < KMPB_COPY_STREAMS; i++) {
        ctx->d_mark[i].release();
        ctx->d_sel_flags[i].release();
        ctx->h_sel_flags[i].release();
        ctx->d_find_rec[i].release();
        ctx->d_stage_bytes[i].release();
        ctx->d_stage_off[i].release();
        ctx->h_stage_bytes[i].release();
        ctx->h_stage_off[i].release();
        if (ctx->ev_h2d[i]) cudaEventDestroy(ctx->ev_h2d[i]);
        if (ctx->copy_stream[i]) cudaStreamDestroy(ctx->copy_stream[i]);
    }
    for (auto &ev : ctx->ev) if (ev) cudaEventDestroy(ev);
    for (auto &ev : ctx->ev_kernel) if (ev) cudaEventDestroy(ev);
    if (ctx->ev_dev) cudaEventDestroy(ctx->ev_dev);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}

int kmpb_set_engine(kmpb_ctx *ctx, int engine)
{
    if (ctx == nullptr) return kmpb_fail(KMPB_EINVAL, "NULL context");
    if (engine != KMPB_ENGINE_AUTO && engine != KMPB_ENGINE_PERPAT && engine != KMPB_ENGINE_UNION)
        return kmpb_fail(KMPB_EINVAL, "unknown engine %d", engine);
    ctx->engine = engine;
    return KMPB_OK;
}

int kmpb_get_device(const kmpb_ctx *ctx) { return ctx ? ctx->device : -1; }
uint64_t *kmpb_device_counts(kmpb_ctx *ctx) { return ctx ? ctx->d_counts : nullptr; }
uint32_t kmpb_pattern_count(const kmpb_ctx *ctx) { return ctx && ctx->have_tables ? ctx->host.n_pat : 0; }
uint64_t kmpb_launch_count(const kmpb_ctx *ctx) { return ctx ? ctx->launches : 0; }

int kmpb_set_profile(kmpb_ctx *ctx, int on)
{
    if (ctx == nullptr) return kmpb_fail(KMPB_EINVAL, "NULL context");
    ctx->profile = on != 0;
    return KMPB_OK;
}

int kmpb_last_kernel_ms(kmpb_ctx *ctx, double *ms_out)
{
    if (ctx == nullptr || ms_out == nullptr) return kmpb_fail(KMPB_EINVAL, "NULL argument");
    if (!ctx->profile) return kmpb_fail(KMPB_ESTATE, "kmpb_set_profile(ctx, 1) first");
    KMPB_CUDA(cudaSetDevice(ctx->device));
    KMPB_CUDA(cudaEventSynchronize(ctx->ev_kernel[1]));
    float ms = 0;
    KMPB_CUDA(cudaEventElapsedTime(&ms, ctx->ev_kernel[0], ctx->ev_kernel[1]));
    *ms_out = ms;
    return KMPB_OK;
}

int kmpb_last_timing(const kmpb_ctx *ctx, double *ms_out, int n)
{
    if (ctx == nullptr || ms_out == nullptr) return kmpb_fail(KMPB_EINVAL, "NULL argument");
    for (int i = 0; i < n && i < 2; i++) ms_out[i] = ctx->last_ms[i];
    return KMPB_OK;
}

int kmpb_set_patterns(kmpb_ctx *ctx, const uint8_t *blob, const uint32_t *pat_off, uint32_t n_pat)
{
    return kmpb_set_patterns_ex(ctx, blob, pat_off, n_pat, nullptr);
}

int kmpb_set_patterns_ex(kmpb_ctx *ctx, const uint8_t *blob, const uint32_t *pat_off, uint32_t n_pat, const uint8_t *flags)
{
    return kmpb_set_patterns_win(ctx, blob, pat_off, n_pat, flags, nullptr);
}

int kmpb_set_patterns_win(kmpb_ctx *ctx, const uint8_t *blob, const uint32_t *pat_off, uint32_t n_pat, const uint8_t *flags,
                          const kmpb_window *win)
{
    if (ctx == nullptr) return kmpb_fail(KMPB_EINVAL, "NULL context");
    int rc = no_open_stream(ctx, "kmpb_set_patterns");
    if (rc || (rc = use_device(ctx))) return rc;
    kmpb_tables fresh;
    rc = kmpb_tables_build_win(&fresh, blob, pat_off, n_pat, flags, win, 0);
    if (rc) return rc;
    KMPB_CUDA(cudaDeviceSynchronize());
    kmpb_release_tables(ctx);
    ctx->host = fresh;
    ctx->have_tables = true;
    rc = kmpb_upload_tables(ctx);
    if (rc) kmpb_release_tables(ctx);
    return rc;
}

int kmpb_get_prefix(kmpb_ctx *ctx, uint32_t pattern_index, int32_t *pi_out, uint32_t capacity)
{
    if (ctx == nullptr || pi_out == nullptr) return kmpb_fail(KMPB_EINVAL, "NULL argument");
    if (!ctx->have_tables) return kmpb_fail(KMPB_ESTATE, "kmpb_get_prefix before kmpb_set_patterns");
    if (pattern_index >= ctx->host.n_pat) return kmpb_fail(KMPB_EINVAL, "pattern index %u out of range", pattern_index);
    int rc = use_device(ctx);
    if (rc) return rc;
    const uint32_t u = ctx->host.pat_to_uniq[pattern_index];
    const uint32_t m = ctx->host.uniq_len[u];
    if (capacity < m) return kmpb_fail(KMPB_EINVAL, "prefix buffer holds %u entries, pattern has %u", capacity, m);
    KMPB_CUDA(cudaMemcpy(pi_out, ctx->dev.pi + ctx->host.uniq_off[u], m * sizeof(int32_t), cudaMemcpyDeviceToHost));
    return KMPB_OK;
}

// Device-resident batch with the byte span given by the caller: fully asynchronous.  The counts are added to
// n_vectors count vectors (this GPU's and/or NVLink-mapped peers'); with the union engine the kernel's
// last block does that itself, so a pass is two launches (work partition, match) and no collective.
static int count_device_span_into(kmpb_ctx *ctx, const uint8_t *d_bytes, const uint64_t *d_offsets, uint64_t n_packets,
                                  uint64_t first_byte, uint64_t end_byte, uint64_t *const *d_counts, uint32_t n_vectors,
                                  void *stream_v, const char *call)
{
    if (ctx == nullptr) return kmpb_fail(KMPB_EINVAL, "NULL context");
    if (int rc = no_open_stream(ctx, call)) return rc;
    if (!ctx->have_tables) return kmpb_fail(KMPB_ESTATE, "count before kmpb_set_patterns");
    if (ctx->host.n_pat == 0) return KMPB_OK;
    if (d_counts == nullptr || n_vectors == 0 || n_vectors > (uint32_t)KMPB_MAX_OUT)
        return kmpb_fail(KMPB_EINVAL, "1..%d count vectors expected", KMPB_MAX_OUT);
    for (uint32_t r = 0; r < n_vectors; r++)
        if (d_counts[r] == nullptr) return kmpb_fail(KMPB_EINVAL, "NULL device pointer");
    if (n_packets && (d_bytes == nullptr || d_offsets == nullptr)) return kmpb_fail(KMPB_EINVAL, "NULL device pointer");
    if (end_byte < first_byte) return kmpb_fail(KMPB_EINVAL, "offsets decrease");
    int rc = use_device(ctx);
    if (rc) return rc;
    cudaStream_t stream = (cudaStream_t)stream_v; // NULL is CUDA's default stream, as in the runtime API
    if ((rc = kmpb_union_scratch(ctx, end_byte - first_byte))) return rc;
    const uint32_t nu = ctx->host.n_uniq;
    kmpb_batch b{d_bytes, 0, d_offsets, n_packets, first_byte, end_byte};
    const bool fused = ctx->engine != KMPB_ENGINE_PERPAT && n_packets > 0 && end_byte > first_byte && nu > 0;
    return device_ordered(ctx, stream, [&]() -> int {
        KMPB_CUDA(cudaMemsetAsync(ctx->d_uniq_counts, 0, (size_t)nu * sizeof(uint64_t), stream));
        if (fused) {
            kmpb_fused_out out;
            out.n = n_vectors;
            for (uint32_t r = 0; r < n_vectors; r++) out.vec[r] = (unsigned long long *)d_counts[r];
            return kmpb_launch_union(ctx, b, 0, ctx->d_uniq_counts, stream, out);
        }
        int rc2 = run_engine(ctx, b, 0, stream);
        if (rc2) return rc2;
        for (uint32_t r = 0; r < n_vectors; r++) {
            kmpb_expand_counts_kernel<<<(ctx->host.n_pat + 255) / 256, 256, 0, stream>>>(
                (const unsigned long long *)ctx->d_uniq_counts, nu, 1, ctx->dev.pat_to_uniq, ctx->host.n_pat,
                (unsigned long long *)d_counts[r], n_vectors > 1 ? 2 : 1);
            ctx->launches++;
        }
        KMPB_CUDA(cudaGetLastError());
        return KMPB_OK;
    });
}

int kmpb_count_device_span(kmpb_ctx *ctx, const uint8_t *d_bytes, const uint64_t *d_offsets, uint64_t n_packets,
                           uint64_t first_byte, uint64_t end_byte, uint64_t *d_counts, void *stream_v)
{
    uint64_t *one[1] = {d_counts};
    return count_device_span_into(ctx, d_bytes, d_offsets, n_packets, first_byte, end_byte, one, 1, stream_v,
                                  "kmpb_count_device_span");
}

int kmpb_count_device_span_peers(kmpb_ctx *ctx, const uint8_t *d_bytes, const uint64_t *d_offsets, uint64_t n_packets,
                                 uint64_t first_byte, uint64_t end_byte, uint64_t *const *d_counts_all,
                                 uint32_t n_vectors, void *stream_v)
{
    return count_device_span_into(ctx, d_bytes, d_offsets, n_packets, first_byte, end_byte, d_counts_all, n_vectors, stream_v,
                                  "kmpb_count_device_span_peers");
}

// (the span read touches only the caller's offsets: the ordering after earlier device-form calls starts in
// kmpb_count_device_span, so the host waits for this call's stream alone, as before)
int kmpb_count_device(kmpb_ctx *ctx, const uint8_t *d_bytes, const uint64_t *d_offsets, uint64_t n_packets,
                      uint64_t *d_counts, void *stream_v)
{
    if (ctx == nullptr) return kmpb_fail(KMPB_EINVAL, "NULL context");
    if (int rc = no_open_stream(ctx, "kmpb_count_device")) return rc;
    if (n_packets == 0) return KMPB_OK;
    if (d_offsets == nullptr) return kmpb_fail(KMPB_EINVAL, "NULL device pointer");
    int rc = use_device(ctx);
    if (rc) return rc;
    cudaStream_t stream = (cudaStream_t)stream_v;
    uint64_t span[2];
    KMPB_CUDA(cudaMemcpyAsync(&span[0], d_offsets, sizeof(uint64_t), cudaMemcpyDeviceToHost, stream));
    KMPB_CUDA(cudaMemcpyAsync(&span[1], d_offsets + n_packets, sizeof(uint64_t), cudaMemcpyDeviceToHost, stream));
    KMPB_CUDA(cudaStreamSynchronize(stream));
    return kmpb_count_device_span(ctx, d_bytes, d_offsets, n_packets, span[0], span[1], d_counts, stream_v);
}

int kmpb_count_host(kmpb_ctx *ctx, const uint8_t *bytes, const uint64_t *offsets, uint64_t n_packets,
                    uint64_t *counts_out)
{
    host_input in{bytes, offsets, n_packets};
    return count_chunked(ctx, in, counts_out, "kmpb_count_host");
}

int kmpb_reserve_staging(kmpb_ctx *ctx, uint64_t max_batch_bytes, uint64_t max_packets)
{
    if (ctx == nullptr) return kmpb_fail(KMPB_EINVAL, "NULL argument");
    int rc = no_open_stream(ctx, "kmpb_reserve_staging");
    if (rc) return rc;
    if (max_batch_bytes == 0) max_batch_bytes = (64ull << 20) + 65536; // a ~64 MiB batch of whole packets
    if (max_packets == 0) max_packets = 1ull << 20;
    if ((rc = use_device(ctx))) return rc;
    return reserve(ctx, max_batch_bytes, max_packets, true);
}

int kmpb_count_pcap(kmpb_ctx *ctx, const kmpb_pcap *pc, uint64_t first, uint64_t count, uint64_t *counts_out)
{
    if (ctx == nullptr || pc == nullptr) return kmpb_fail(KMPB_EINVAL, "NULL argument");
    pcap_input in{pc, first, count};
    return count_chunked(ctx, in, counts_out, "kmpb_count_pcap");
}

// ---- find: where the patterns occur (include/kmpb200.h; kernels in union_kernel.cu and find.cu) ----------------
int kmpb_find_device_span(kmpb_ctx *ctx, const uint8_t *d_bytes, const uint64_t *d_offsets, uint64_t n_packets,
                          uint64_t first_byte, uint64_t end_byte, kmpb_match *d_out, uint64_t capacity,
                          uint64_t *d_n_found, uint32_t flags, void *stream_v)
{
    int rc = find_args(ctx, d_out, capacity, d_n_found, "kmpb_find_device_span");
    if (rc) return rc;
    if (flags & ~KMPB_FIND_SORTED) return kmpb_fail(KMPB_EINVAL, "unknown find flags 0x%x", flags);
    if (n_packets && (d_bytes == nullptr || d_offsets == nullptr)) return kmpb_fail(KMPB_EINVAL, "NULL device pointer");
    if (end_byte < first_byte) return kmpb_fail(KMPB_EINVAL, "offsets decrease");
    if ((rc = use_device(ctx))) return rc;
    cudaStream_t stream = (cudaStream_t)stream_v;
    if ((rc = kmpb_union_scratch(ctx, end_byte - first_byte))) return rc;
    const kmpb_batch b{d_bytes, 0, d_offsets, n_packets, first_byte, end_byte};
    unsigned long long *found = reinterpret_cast<unsigned long long *>(d_n_found);
    return device_ordered(ctx, stream, [&]() -> int {
        const int rc2 = kmpb_find_match(ctx, b, 0, d_out, capacity, found, stream);
        return rc2 ? rc2 : kmpb_find_finish(ctx, b, 0, d_out, capacity, found, (flags & KMPB_FIND_SORTED) != 0, stream);
    });
}

int kmpb_find_host(kmpb_ctx *ctx, const uint8_t *bytes, const uint64_t *offsets, uint64_t n_packets,
                   kmpb_match *out, uint64_t capacity, uint64_t *n_found)
{
    host_input in{bytes, offsets, n_packets};
    return find_chunked(ctx, in, out, capacity, n_found, "kmpb_find_host");
}

int kmpb_find_pcap(kmpb_ctx *ctx, const kmpb_pcap *pc, uint64_t first, uint64_t count, kmpb_match *out, uint64_t capacity,
                   uint64_t *n_found)
{
    if (pc == nullptr) return kmpb_fail(KMPB_EINVAL, "NULL argument");
    pcap_input in{pc, first, count};
    return find_chunked(ctx, in, out, capacity, n_found, "kmpb_find_pcap");
}

// ---- select: which packets match (include/kmpb200.h; kernels in union_kernel.cu and select.cu) ------------------
int kmpb_select_device_span(kmpb_ctx *ctx, const uint8_t *d_bytes, const uint64_t *d_offsets, uint64_t n_packets,
                            uint64_t first_byte, uint64_t end_byte, uint8_t *d_flags, uint64_t *d_index,
                            uint64_t *d_n_selected, uint64_t *d_counts, uint32_t flags, void *stream_v)
{
    int rc = select_args(ctx, d_flags, n_packets, "kmpb_select_device_span");
    if (rc) return rc;
    if (flags & ~KMPB_SELECT_INVERT) return kmpb_fail(KMPB_EINVAL, "unknown select flags 0x%x", flags);
    if (d_index && !d_n_selected) return kmpb_fail(KMPB_EINVAL, "d_index without d_n_selected");
    if (n_packets && (d_bytes == nullptr || d_offsets == nullptr)) return kmpb_fail(KMPB_EINVAL, "NULL device pointer");
    if (end_byte < first_byte) return kmpb_fail(KMPB_EINVAL, "offsets decrease");
    if ((rc = use_device(ctx))) return rc;
    cudaStream_t stream = (cudaStream_t)stream_v;
    if ((rc = kmpb_union_scratch(ctx, end_byte - first_byte))) return rc;
    const kmpb_batch b{d_bytes, 0, d_offsets, n_packets, first_byte, end_byte};
    kmpb_fused_out out;
    out.n = d_counts ? 1 : 0;
    out.vec[0] = reinterpret_cast<unsigned long long *>(d_counts);
    return device_ordered(ctx, stream, [&]() -> int {
        if (ctx->host.n_uniq) KMPB_CUDA(cudaMemsetAsync(ctx->d_uniq_counts, 0, (size_t)ctx->host.n_uniq * sizeof(uint64_t), stream));
        int rc2 = kmpb_select_match(ctx, b, 0, d_flags, stream, out);
        if (rc2 || !d_n_selected) return rc2;
        return kmpb_select_compact(ctx, d_flags, n_packets, (flags & KMPB_SELECT_INVERT) != 0, d_index, d_n_selected, stream);
    });
}

int kmpb_select_host(kmpb_ctx *ctx, const uint8_t *bytes, const uint64_t *offsets, uint64_t n_packets, uint8_t *flags_out,
                     uint64_t *n_selected, uint64_t *counts_out)
{
    host_input in{bytes, offsets, n_packets};
    return select_chunked(ctx, in, flags_out, n_selected, counts_out, "kmpb_select_host");
}

int kmpb_select_pcap(kmpb_ctx *ctx, const kmpb_pcap *pc, uint64_t first, uint64_t count, uint8_t *flags_out,
                     uint64_t *n_selected, uint64_t *counts_out)
{
    if (pc == nullptr) return kmpb_fail(KMPB_EINVAL, "NULL argument");
    pcap_input in{pc, first, count};
    return select_chunked(ctx, in, flags_out, n_selected, counts_out, "kmpb_select_pcap");
}

// ---- frames pushed one at a time (the live-capture shape) ----------------------------------------
struct kmpb_stream {
    kmpb_ctx *ctx;
    int (*extract)(const uint8_t *, uint32_t, uint32_t *, uint32_t *);
    uint64_t batch_bytes, max_pkts;
    int slot;            // staging slot being filled
    uint64_t n, bytes;   // packets and payload bytes in it
    uint64_t batches, frames, packets;
};

static int stream_submit(kmpb_stream *st)
{
    kmpb_ctx *ctx = st->ctx;
    if (st->n == 0) return KMPB_OK;
    const int slot = st->slot;
    ctx->h_stage_off[slot].p[st->n] = st->bytes;
    kmpb_batch b;
    int rc;
    if ((rc = submit_pinned(ctx, slot, st->n, st->bytes, b)) ||
        (rc = run_engine(ctx, b, slot, ctx->copy_stream[slot]))) // accumulates into the slot's distinct-pattern counters
        return rc;
    st->batches++;
    st->slot = (slot + 1) % KMPB_COPY_STREAMS;
    st->n = st->bytes = 0;
    return wait_pinned(ctx, st->slot); // kmpb_stream_push fills it next
}

int kmpb_stream_open(kmpb_ctx *ctx, int proto, uint64_t batch_bytes, kmpb_stream **out)
{
    if (ctx == nullptr || out == nullptr) return kmpb_fail(KMPB_EINVAL, "NULL argument");
    *out = nullptr;
    int rc = no_open_stream(ctx, "kmpb_stream_open");
    if (rc) return rc;
    if (!ctx->have_tables) return kmpb_fail(KMPB_ESTATE, "stream before kmpb_set_patterns");
    if (proto != KMPB_PROTO_UDP && proto != KMPB_PROTO_TCP) return kmpb_fail(KMPB_EINVAL, "unknown protocol %d", proto);
    if ((rc = use_device(ctx))) return rc;
    if (batch_bytes == 0) batch_bytes = 8ull << 20;
    if (batch_bytes < 65536) batch_bytes = 65536; // a frame's payload is at most 65535 - headers bytes long... jumbo included
    const uint64_t max_pkts = 1ull << 20;
    if ((rc = reserve(ctx, batch_bytes, max_pkts, true)) || (rc = start_chunks(ctx, KMPB_COPY_STREAMS))) return rc;
    KMPB_CUDA(cudaStreamSynchronize(ctx->stream));
    kmpb_stream *st = new (std::nothrow) kmpb_stream();
    if (st == nullptr) return kmpb_fail(KMPB_ENOMEM, "out of memory");
    st->ctx = ctx;
    st->extract = proto == KMPB_PROTO_TCP ? kmpb_extract_tcp : kmpb_extract_udp;
    st->batch_bytes = batch_bytes;
    st->max_pkts = max_pkts;
    st->slot = 0;
    st->n = st->bytes = st->batches = st->frames = st->packets = 0;
    ctx->open_streams++;
    *out = st;
    return KMPB_OK;
}

int kmpb_stream_push(kmpb_stream *st, const uint8_t *frame, uint32_t captured_len)
{
    if (st == nullptr || (frame == nullptr && captured_len)) return kmpb_fail(KMPB_EINVAL, "NULL argument");
    uint32_t off = 0, len = 0;
    st->frames++;
    if (!st->extract(frame, captured_len, &off, &len)) return KMPB_OK;
    if (len >= KMPB_PACKET_LIMIT)
        return kmpb_fail(KMPB_ELIMIT, "packet %llu has a payload of %u bytes; packets must be shorter than %llu (2 GiB - 1 MiB)",
                         (unsigned long long)st->packets, len, KMPB_PACKET_LIMIT);
    if (len > st->batch_bytes) return kmpb_fail(KMPB_ELIMIT, "a %u-byte payload does not fit a %llu-byte batch", len, (unsigned long long)st->batch_bytes);
    int rc = use_device(st->ctx);
    if (rc) return rc;
    if (st->bytes + len > st->batch_bytes || st->n == st->max_pkts)
        if ((rc = stream_submit(st))) return rc;
    kmpb_ctx *ctx = st->ctx;
    ctx->h_stage_off[st->slot].p[st->n] = st->bytes;
    memcpy(ctx->h_stage_bytes[st->slot].p + st->bytes, frame + off, len);
    st->n++;
    st->bytes += len;
    st->packets++;
    return KMPB_OK;
}

int kmpb_stream_flush(kmpb_stream *st, uint64_t *counts_out)
{
    if (st == nullptr || counts_out == nullptr) return kmpb_fail(KMPB_EINVAL, "NULL argument");
    kmpb_ctx *ctx = st->ctx;
    if (ctx->host.n_pat == 0) return KMPB_OK;
    int rc = use_device(ctx);
    if (rc) return rc;
    if ((rc = stream_submit(st))) return rc;
    return finish_chunked(ctx, KMPB_COPY_STREAMS, counts_out);
}

uint64_t kmpb_stream_packets(const kmpb_stream *st) { return st ? st->packets : 0; }

void kmpb_stream_close(kmpb_stream *st)
{
    if (st == nullptr) return;
    cudaSetDevice(st->ctx->device);
    cudaDeviceSynchronize();
    st->ctx->open_streams--;
    delete st;
}

void *kmpb_host_alloc(size_t bytes)
{
    void *p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocDefault) != cudaSuccess) {
        cudaGetLastError();
        kmpb_fail(KMPB_ENOMEM, "cudaHostAlloc(%zu) failed", bytes);
        return nullptr;
    }
    return p;
}

void kmpb_host_free(void *p)
{
    if (p) cudaFreeHost(p);
}

} // extern "C"
