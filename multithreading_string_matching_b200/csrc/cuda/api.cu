// api.cu -- the C ABI of include/kmpb200.h: context, pattern upload, the two count entry points.
#include <algorithm>
#include <new>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>
#include <vector>

#include "kmpb_device.cuh"

// a CUDA call inside a chunk loop: on failure nothing of the call stays in flight
#define KMPB_CUDA_Q(ctx, call)                                                                   \
    do {                                                                                         \
        cudaError_t e_ = (call);                                                                 \
        if (e_ != cudaSuccess) {                                                                 \
            quiesce(ctx);                                                                        \
            return kmpb_fail(KMPB_ECUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), \
                             __FILE__, __LINE__);                                                \
        }                                                                                        \
    } while (0)

namespace {

void quiesce(kmpb_ctx *ctx);

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

// device staging slots for chunked host input (grown on demand, kept for the next call)
int ensure_staging(kmpb_ctx *ctx, uint64_t max_bytes, uint64_t max_pkts)
{
    if (max_bytes + 1024 <= ctx->stage_bytes_cap && max_pkts + 1 <= ctx->stage_off_cap) return KMPB_OK;
    KMPB_CUDA(cudaDeviceSynchronize());
    const size_t bcap = std::max<size_t>(ctx->stage_bytes_cap, (size_t)max_bytes + 1024);
    const size_t ocap = std::max<size_t>(ctx->stage_off_cap, (size_t)max_pkts + 1);
    for (int i = 0; i < KMPB_COPY_STREAMS; i++) {
        cudaFree(ctx->d_stage_bytes[i]); ctx->d_stage_bytes[i] = nullptr;
        cudaFree(ctx->d_stage_off[i]); ctx->d_stage_off[i] = nullptr;
    }
    ctx->stage_bytes_cap = ctx->stage_off_cap = 0;
    for (int i = 0; i < KMPB_COPY_STREAMS; i++) {
        KMPB_CUDA(cudaMalloc((void **)&ctx->d_stage_bytes[i], bcap));
        KMPB_CUDA(cudaMemset(ctx->d_stage_bytes[i], 0, bcap));
        KMPB_CUDA(cudaMalloc((void **)&ctx->d_stage_off[i], ocap * sizeof(uint64_t)));
    }
    ctx->stage_bytes_cap = bcap;
    ctx->stage_off_cap = ocap;
    return KMPB_OK;
}

// ... and their pinned twins on the host
int ensure_host_staging(kmpb_ctx *ctx, uint64_t max_bytes, uint64_t max_pkts)
{
    if (max_bytes + 1024 <= ctx->h_stage_bytes_cap && max_pkts + 1 <= ctx->h_stage_off_cap) return KMPB_OK;
    KMPB_CUDA(cudaDeviceSynchronize());
    const size_t bcap = std::max<size_t>(ctx->h_stage_bytes_cap, (size_t)max_bytes + 1024);
    const size_t ocap = std::max<size_t>(ctx->h_stage_off_cap, (size_t)max_pkts + 1);
    for (int i = 0; i < KMPB_COPY_STREAMS; i++) {
        cudaFreeHost(ctx->h_stage_bytes[i]); ctx->h_stage_bytes[i] = nullptr;
        cudaFreeHost(ctx->h_stage_off[i]); ctx->h_stage_off[i] = nullptr;
    }
    ctx->h_stage_bytes_cap = ctx->h_stage_off_cap = 0;
    for (int i = 0; i < KMPB_COPY_STREAMS; i++) {
        KMPB_CUDA(cudaHostAlloc((void **)&ctx->h_stage_bytes[i], bcap, cudaHostAllocDefault));
        KMPB_CUDA(cudaHostAlloc((void **)&ctx->h_stage_off[i], ocap * sizeof(uint64_t), cudaHostAllocDefault));
        if (!ctx->ev_h2d[i]) KMPB_CUDA(cudaEventCreateWithFlags(&ctx->ev_h2d[i], cudaEventDisableTiming));
    }
    ctx->h_stage_bytes_cap = bcap;
    ctx->h_stage_off_cap = ocap;
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

// chunk plan of a host batch: whole packets, ~chunk_bytes each; the largest chunk's bytes (from its 512-byte aligned
// base) and packets
struct host_chunk { uint64_t k0, k1; };
std::vector<host_chunk> plan_host_chunks(const uint64_t *offsets, uint64_t n_packets, uint64_t chunk_bytes, uint64_t &max_bytes,
                                         uint64_t &max_pkts)
{
    std::vector<host_chunk> plan;
    max_bytes = max_pkts = 0;
    for (uint64_t k0 = 0; k0 < n_packets;) {
        const uint64_t want = offsets[k0] + chunk_bytes;
        uint64_t k1 = (uint64_t)(std::lower_bound(offsets + k0 + 1, offsets + n_packets, want) - offsets);
        if (k1 > n_packets) k1 = n_packets;
        k1 = std::min<uint64_t>(k1, k0 + ((1ull << 31) - 2));
        plan.push_back({k0, k1});
        const uint64_t base = offsets[k0] & ~511ull;
        max_bytes = std::max(max_bytes, offsets[k1] - base);
        max_pkts = std::max(max_pkts, k1 - k0);
        k0 = k1;
    }
    return plan;
}

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

// the record buffer of a stream slot of the chunked find forms, at least `records` long (grown by an eighth more)
int ensure_find_rec(kmpb_ctx *ctx, int slot, uint64_t records)
{
    if (!ctx->d_find_found) KMPB_CUDA(cudaMalloc((void **)&ctx->d_find_found, KMPB_COPY_STREAMS * sizeof(unsigned long long)));
    if (records <= ctx->find_rec_cap[slot] && ctx->d_find_rec[slot]) return KMPB_OK;
    const uint64_t cap = records + records / 8 + 1024;
    cudaFree(ctx->d_find_rec[slot]);
    ctx->d_find_rec[slot] = nullptr;
    ctx->find_rec_cap[slot] = 0;
    KMPB_CUDA(cudaMalloc((void **)&ctx->d_find_rec[slot], cap * sizeof(kmpb_match)));
    ctx->find_rec_cap[slot] = cap;
    return KMPB_OK;
}

// The chunk pipeline of the host find forms.  stage(c, slot, batch, packet_base) puts chunk c on the device in the
// slot's staging buffers (copies on the slot's stream) -- kmpb_count_host's or kmpb_count_pcap's way; the find kernel
// follows on the same stream.  Chunk c is finished (its match count read, its records sorted and copied out) just
// before its slot takes chunk c + KMPB_COPY_STREAMS, so the copies and kernels of the chunks in between keep the device
// busy meanwhile.  A chunk whose records overflowed the slot's buffer is matched again, from the copy still on the
// device, into a buffer of the exact size; once `capacity` records are out, later chunks are only counted.
template <class Stage>
int find_chunks(kmpb_ctx *ctx, uint64_t n_chunks, uint64_t guess, Stage &&stage, kmpb_match *out, uint64_t capacity,
                uint64_t *n_found)
{
    kmpb_batch batch[KMPB_COPY_STREAMS] = {};
    uint64_t base[KMPB_COPY_STREAMS] = {};
    uint64_t total = 0, written = 0;
    int rc;
    auto finish = [&](uint64_t c) -> int {
        const int slot = (int)(c % KMPB_COPY_STREAMS);
        cudaStream_t s = ctx->copy_stream[slot];
        unsigned long long n = 0;
        KMPB_CUDA_Q(ctx, cudaMemcpyAsync(&n, ctx->d_find_found + slot, sizeof n, cudaMemcpyDeviceToHost, s));
        KMPB_CUDA_Q(ctx, cudaStreamSynchronize(s));
        const uint64_t take = std::min<uint64_t>(n, capacity - written);
        if (take) {
            int rc2;
            if (n > ctx->find_rec_cap[slot]) {
                if ((rc2 = ensure_find_rec(ctx, slot, n)) || (rc2 = kmpb_find_match(ctx, batch[slot], slot, ctx->d_find_rec[slot], n,
                                                                                     ctx->d_find_found + slot, s))) {
                    quiesce(ctx);
                    return rc2;
                }
            }
            if ((rc2 = kmpb_find_finish(ctx, batch[slot], base[slot], ctx->d_find_rec[slot], n, ctx->d_find_found + slot, true, s))) {
                quiesce(ctx);
                return rc2;
            }
            KMPB_CUDA_Q(ctx, cudaMemcpyAsync(out + written, ctx->d_find_rec[slot], take * sizeof(kmpb_match), cudaMemcpyDeviceToHost, s));
            KMPB_CUDA_Q(ctx, cudaStreamSynchronize(s));
        }
        total += n;
        written += take;
        return KMPB_OK;
    };
    for (uint64_t c = 0; c < n_chunks; c++) {
        const int slot = (int)(c % KMPB_COPY_STREAMS);
        if (c >= (uint64_t)KMPB_COPY_STREAMS && (rc = finish(c - KMPB_COPY_STREAMS))) return rc;
        if ((rc = ensure_find_rec(ctx, slot, guess))) { quiesce(ctx); return rc; }
        if ((rc = stage(c, slot, batch[slot], base[slot])) ||
            (rc = kmpb_find_match(ctx, batch[slot], slot, ctx->d_find_rec[slot], ctx->find_rec_cap[slot], ctx->d_find_found + slot,
                                  ctx->copy_stream[slot]))) {
            quiesce(ctx);
            return rc;
        }
    }
    for (uint64_t c = n_chunks > (uint64_t)KMPB_COPY_STREAMS ? n_chunks - KMPB_COPY_STREAMS : 0; c < n_chunks; c++)
        if ((rc = finish(c))) return rc;
    *n_found = total;
    return KMPB_OK; // (as in finish_chunked: the stage's caller checked every packet's size first)
}

// the argument checks every find form starts with
int find_args(kmpb_ctx *ctx, const void *out, uint64_t capacity, const void *n_found)
{
    if (ctx == nullptr || n_found == nullptr || (out == nullptr && capacity)) return kmpb_fail(KMPB_EINVAL, "NULL argument");
    if (!ctx->have_tables) return kmpb_fail(KMPB_ESTATE, "find before kmpb_set_patterns");
    return KMPB_OK;
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
    if (ctx->d_work == nullptr) return KMPB_OK;
    // the union engine's error flags, word 1 of every slot's work counters: set by its kernels, cleared only here
    uint32_t work[KMPB_COPY_STREAMS * 4];
    KMPB_CUDA(cudaMemcpy(work, ctx->d_work, sizeof work, cudaMemcpyDeviceToHost));
    bool flagged = false;
    for (int s = 0; s < KMPB_COPY_STREAMS; s++) flagged |= work[s * 4 + 1] != 0;
    if (!flagged) return KMPB_OK;
    KMPB_CUDA(cudaMemset(ctx->d_work, 0, sizeof work));
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
    cudaFree(ctx->d_work);
    cudaFree(ctx->d_items);
    cudaFree(ctx->d_find_found);
    cudaFree(ctx->d_sort_keys[0]);
    cudaFree(ctx->d_sort_keys[1]);
    cudaFree(ctx->d_sort_temp);
    for (int i = 0; i < KMPB_COPY_STREAMS; i++) {
        cudaFree(ctx->d_find_rec[i]);
        cudaFree(ctx->d_stage_bytes[i]);
        cudaFree(ctx->d_stage_off[i]);
        cudaFreeHost(ctx->h_stage_bytes[i]);
        cudaFreeHost(ctx->h_stage_off[i]);
        if (ctx->ev_h2d[i]) cudaEventDestroy(ctx->ev_h2d[i]);
        if (ctx->copy_stream[i]) cudaStreamDestroy(ctx->copy_stream[i]);
    }
    for (auto &ev : ctx->ev) if (ev) cudaEventDestroy(ev);
    for (auto &ev : ctx->ev_kernel) if (ev) cudaEventDestroy(ev);
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
    if (ctx == nullptr) return kmpb_fail(KMPB_EINVAL, "NULL context");
    int rc = use_device(ctx);
    if (rc) return rc;
    kmpb_tables fresh;
    rc = kmpb_tables_build(&fresh, blob, pat_off, n_pat);
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
                                  void *stream_v)
{
    if (ctx == nullptr) return kmpb_fail(KMPB_EINVAL, "NULL context");
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
    KMPB_CUDA(cudaMemsetAsync(ctx->d_uniq_counts, 0, (size_t)nu * sizeof(uint64_t), stream));
    kmpb_batch b{d_bytes, 0, d_offsets, n_packets, first_byte, end_byte};
    const bool fused = ctx->engine != KMPB_ENGINE_PERPAT && n_packets > 0 && end_byte > first_byte && nu > 0;
    if (fused) {
        kmpb_fused_out out;
        out.n = n_vectors;
        for (uint32_t r = 0; r < n_vectors; r++) out.vec[r] = (unsigned long long *)d_counts[r];
        return kmpb_launch_union(ctx, b, 0, ctx->d_uniq_counts, stream, out);
    }
    if ((rc = run_engine(ctx, b, 0, stream))) return rc;
    for (uint32_t r = 0; r < n_vectors; r++) {
        kmpb_expand_counts_kernel<<<(ctx->host.n_pat + 255) / 256, 256, 0, stream>>>(
            (const unsigned long long *)ctx->d_uniq_counts, nu, 1, ctx->dev.pat_to_uniq, ctx->host.n_pat,
            (unsigned long long *)d_counts[r], n_vectors > 1 ? 2 : 1);
        ctx->launches++;
    }
    KMPB_CUDA(cudaGetLastError());
    return KMPB_OK;
}

int kmpb_count_device_span(kmpb_ctx *ctx, const uint8_t *d_bytes, const uint64_t *d_offsets, uint64_t n_packets,
                           uint64_t first_byte, uint64_t end_byte, uint64_t *d_counts, void *stream_v)
{
    uint64_t *one[1] = {d_counts};
    return count_device_span_into(ctx, d_bytes, d_offsets, n_packets, first_byte, end_byte, one, 1, stream_v);
}

int kmpb_count_device_span_peers(kmpb_ctx *ctx, const uint8_t *d_bytes, const uint64_t *d_offsets, uint64_t n_packets,
                                 uint64_t first_byte, uint64_t end_byte, uint64_t *const *d_counts_all,
                                 uint32_t n_vectors, void *stream_v)
{
    return count_device_span_into(ctx, d_bytes, d_offsets, n_packets, first_byte, end_byte, d_counts_all, n_vectors, stream_v);
}

int kmpb_count_device(kmpb_ctx *ctx, const uint8_t *d_bytes, const uint64_t *d_offsets, uint64_t n_packets,
                      uint64_t *d_counts, void *stream_v)
{
    if (ctx == nullptr) return kmpb_fail(KMPB_EINVAL, "NULL context");
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

// Host batch: chunks of whole packets are copied to per-stream staging buffers and matched there, so
// the H2D copy of chunk c+1.. overlaps the kernels of chunk c (the MPI variant's Scatterv, done by
// the copy engines instead of the network: mpi_dumping.c:161).
int kmpb_count_host(kmpb_ctx *ctx, const uint8_t *bytes, const uint64_t *offsets, uint64_t n_packets,
                    uint64_t *counts_out)
{
    if (ctx == nullptr) return kmpb_fail(KMPB_EINVAL, "NULL context");
    if (!ctx->have_tables) return kmpb_fail(KMPB_ESTATE, "count before kmpb_set_patterns");
    const uint32_t n_pat = ctx->host.n_pat, nu = ctx->host.n_uniq;
    if (n_pat == 0) return KMPB_OK;
    if (counts_out == nullptr) return kmpb_fail(KMPB_EINVAL, "NULL counts_out");
    memset(counts_out, 0, (size_t)n_pat * sizeof(uint64_t));
    if (n_packets == 0) return KMPB_OK;
    if (bytes == nullptr || offsets == nullptr) return kmpb_fail(KMPB_EINVAL, "NULL batch pointer");
    int rc = check_offsets(offsets, n_packets);
    if (rc) return rc;
    if ((rc = use_device(ctx))) return rc;

    uint64_t max_bytes = 0, max_pkts = 0;
    const std::vector<host_chunk> plan = plan_host_chunks(offsets, n_packets, chunk_bytes_setting(), max_bytes, max_pkts);
    const int n_slots = (int)std::min<size_t>(KMPB_COPY_STREAMS, plan.size());
    if ((rc = ensure_staging(ctx, max_bytes, max_pkts))) return rc;
    if ((rc = kmpb_union_scratch(ctx, max_bytes))) return rc;

    KMPB_CUDA(cudaEventRecord(ctx->ev[0], ctx->stream));
    KMPB_CUDA(cudaMemsetAsync(ctx->d_uniq_counts, 0, (size_t)KMPB_COPY_STREAMS * nu * sizeof(uint64_t), ctx->stream));
    KMPB_CUDA(cudaEventRecord(ctx->ev[2], ctx->stream));
    for (int s = 0; s < n_slots; s++) KMPB_CUDA(cudaStreamWaitEvent(ctx->copy_stream[s], ctx->ev[2], 0));
    for (size_t c = 0; c < plan.size(); c++) {
        const int slot = (int)(c % KMPB_COPY_STREAMS);
        cudaStream_t s = ctx->copy_stream[slot];
        const uint64_t k0 = plan[c].k0, k1 = plan[c].k1;
        const uint64_t base = offsets[k0] & ~511ull;
        KMPB_CUDA_Q(ctx, cudaMemcpyAsync(ctx->d_stage_bytes[slot], bytes + base, offsets[k1] - base, cudaMemcpyHostToDevice, s));
        KMPB_CUDA_Q(ctx, cudaMemcpyAsync(ctx->d_stage_off[slot], offsets + k0, (k1 - k0 + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, s));
        kmpb_batch b{ctx->d_stage_bytes[slot], base, ctx->d_stage_off[slot], k1 - k0, offsets[k0], offsets[k1]};
        if ((rc = run_engine(ctx, b, slot, s))) { quiesce(ctx); return rc; }
    }
    return finish_chunked(ctx, n_slots, counts_out);
}

// Streamed savefile path: pack a chunk of payloads into a pinned staging slot (all host threads), copy
// it to the slot's device twin and match it on the slot's stream while the next chunk is packed -- the
// producer/consumer shape of openmp_task.c:113-178 with the GPU as the consumer.
int kmpb_reserve_staging(kmpb_ctx *ctx, uint64_t max_batch_bytes, uint64_t max_packets)
{
    if (ctx == nullptr) return kmpb_fail(KMPB_EINVAL, "NULL argument");
    if (max_batch_bytes == 0) max_batch_bytes = (64ull << 20) + 65536; // a ~64 MiB batch of whole packets
    if (max_packets == 0) max_packets = 1ull << 20;
    int rc = use_device(ctx);
    if (rc) return rc;
    if ((rc = ensure_staging(ctx, max_batch_bytes, max_packets))) return rc;
    if ((rc = ensure_host_staging(ctx, max_batch_bytes, max_packets))) return rc;
    return kmpb_union_scratch(ctx, max_batch_bytes);
}

int kmpb_count_pcap(kmpb_ctx *ctx, const kmpb_pcap *pc, uint64_t first, uint64_t count, uint64_t *counts_out)
{
    if (ctx == nullptr || pc == nullptr) return kmpb_fail(KMPB_EINVAL, "NULL argument");
    if (!ctx->have_tables) return kmpb_fail(KMPB_ESTATE, "count before kmpb_set_patterns");
    const uint32_t n_pat = ctx->host.n_pat, nu = ctx->host.n_uniq;
    if (n_pat == 0) return KMPB_OK;
    if (counts_out == nullptr) return kmpb_fail(KMPB_EINVAL, "NULL counts_out");
    memset(counts_out, 0, (size_t)n_pat * sizeof(uint64_t));
    const uint64_t total = kmpb_pcap_packets(pc);
    if (first > total || count > total - first) return kmpb_fail(KMPB_EINVAL, "packet range outside the file");
    if (count == 0) return KMPB_OK;
    int rc = check_pcap_lengths(pc, first, count);
    if (rc) return rc;
    if ((rc = use_device(ctx))) return rc;
    if (rc) return rc;
    const uint64_t chunk_bytes = chunk_bytes_setting();
    const uint64_t max_pkts = 1ull << 22, last = first + count;
    // a packet larger than a chunk still travels whole: size the slots for the largest chunk of the plan
    uint64_t max_bytes = 0, max_n = 0, n_chunks = 0;
    for (uint64_t k0 = first; k0 < last; n_chunks++) {
        uint64_t b = 0;
        const uint64_t k1 = kmpb_pcap_chunk_end(pc, k0, last, chunk_bytes, max_pkts, &b);
        max_bytes = std::max(max_bytes, b);
        max_n = std::max(max_n, k1 - k0);
        k0 = k1;
    }
    if ((rc = ensure_staging(ctx, max_bytes, max_n))) return rc;
    if ((rc = ensure_host_staging(ctx, max_bytes, max_n))) return rc;
    if ((rc = kmpb_union_scratch(ctx, max_bytes))) return rc;
    const int n_slots = (int)std::min<uint64_t>(KMPB_COPY_STREAMS, n_chunks);

    KMPB_CUDA(cudaEventRecord(ctx->ev[0], ctx->stream));
    KMPB_CUDA(cudaMemsetAsync(ctx->d_uniq_counts, 0, (size_t)KMPB_COPY_STREAMS * nu * sizeof(uint64_t), ctx->stream));
    KMPB_CUDA(cudaEventRecord(ctx->ev[2], ctx->stream));
    for (int s = 0; s < n_slots; s++) KMPB_CUDA(cudaStreamWaitEvent(ctx->copy_stream[s], ctx->ev[2], 0));
    uint64_t c = 0;
    double t_wait = 0, t_pack = 0, t_issue = 0;
    const bool stats = getenv("KMPB_STATS") != nullptr;
    auto now = []() { timespec ts; clock_gettime(CLOCK_MONOTONIC, &ts); return ts.tv_sec + 1e-9 * ts.tv_nsec; };
    for (uint64_t k0 = first; k0 < last; c++) {
        const int slot = (int)(c % KMPB_COPY_STREAMS);
        cudaStream_t s = ctx->copy_stream[slot];
        uint64_t nbytes = 0;
        const uint64_t k1 = kmpb_pcap_chunk_end(pc, k0, last, chunk_bytes, max_pkts, &nbytes);
        const double t0 = now();
        if (c >= KMPB_COPY_STREAMS) KMPB_CUDA_Q(ctx, cudaEventSynchronize(ctx->ev_h2d[slot])); // the slot's last copy has left it
        const double t1 = now();
        kmpb_pcap_pack(pc, k0, k1 - k0, ctx->h_stage_bytes[slot], ctx->h_stage_off[slot]);
        memset(ctx->h_stage_bytes[slot] + nbytes, 0, 64);
        const double t2 = now();
        KMPB_CUDA_Q(ctx, cudaMemcpyAsync(ctx->d_stage_bytes[slot], ctx->h_stage_bytes[slot], nbytes + 64, cudaMemcpyHostToDevice, s));
        KMPB_CUDA_Q(ctx, cudaMemcpyAsync(ctx->d_stage_off[slot], ctx->h_stage_off[slot], (k1 - k0 + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, s));
        KMPB_CUDA_Q(ctx, cudaEventRecord(ctx->ev_h2d[slot], s));
        kmpb_batch b{ctx->d_stage_bytes[slot], 0, ctx->d_stage_off[slot], k1 - k0, 0, nbytes};
        if ((rc = run_engine(ctx, b, slot, s))) { quiesce(ctx); return rc; }
        k0 = k1;
        t_wait += t1 - t0;
        t_pack += t2 - t1;
        t_issue += now() - t2;
    }
    if (stats)
        fprintf(stderr, "kmpb_count_pcap: %llu chunks; waiting for a free slot %.3f s, packing %.3f s, issuing copies and kernels %.3f s\n",
                (unsigned long long)c, t_wait, t_pack, t_issue);
    return finish_chunked(ctx, n_slots, counts_out);
}

// ---- find: where the patterns occur (include/kmpb200.h; kernels in union_kernel.cu and find.cu) ----------------
int kmpb_find_device_span(kmpb_ctx *ctx, const uint8_t *d_bytes, const uint64_t *d_offsets, uint64_t n_packets,
                          uint64_t first_byte, uint64_t end_byte, kmpb_match *d_out, uint64_t capacity,
                          uint64_t *d_n_found, uint32_t flags, void *stream_v)
{
    int rc = find_args(ctx, d_out, capacity, d_n_found);
    if (rc) return rc;
    if (flags & ~KMPB_FIND_SORTED) return kmpb_fail(KMPB_EINVAL, "unknown find flags 0x%x", flags);
    if (n_packets && (d_bytes == nullptr || d_offsets == nullptr)) return kmpb_fail(KMPB_EINVAL, "NULL device pointer");
    if (end_byte < first_byte) return kmpb_fail(KMPB_EINVAL, "offsets decrease");
    if ((rc = use_device(ctx))) return rc;
    cudaStream_t stream = (cudaStream_t)stream_v;
    if ((rc = kmpb_union_scratch(ctx, end_byte - first_byte))) return rc;
    const kmpb_batch b{d_bytes, 0, d_offsets, n_packets, first_byte, end_byte};
    unsigned long long *found = reinterpret_cast<unsigned long long *>(d_n_found);
    if ((rc = kmpb_find_match(ctx, b, 0, d_out, capacity, found, stream))) return rc;
    return kmpb_find_finish(ctx, b, 0, d_out, capacity, found, (flags & KMPB_FIND_SORTED) != 0, stream);
}

int kmpb_find_host(kmpb_ctx *ctx, const uint8_t *bytes, const uint64_t *offsets, uint64_t n_packets,
                   kmpb_match *out, uint64_t capacity, uint64_t *n_found)
{
    int rc = find_args(ctx, out, capacity, n_found);
    if (rc) return rc;
    *n_found = 0;
    if (ctx->host.n_pat == 0 || n_packets == 0) return KMPB_OK;
    if (bytes == nullptr || offsets == nullptr) return kmpb_fail(KMPB_EINVAL, "NULL batch pointer");
    if ((rc = check_offsets(offsets, n_packets))) return rc;
    if ((rc = use_device(ctx))) return rc;
    uint64_t max_bytes = 0, max_pkts = 0;
    const std::vector<host_chunk> plan = plan_host_chunks(offsets, n_packets, chunk_bytes_setting(), max_bytes, max_pkts);
    if ((rc = ensure_staging(ctx, max_bytes, max_pkts))) return rc;
    if ((rc = kmpb_union_scratch(ctx, max_bytes))) return rc;
    auto stage = [&](uint64_t c, int slot, kmpb_batch &b, uint64_t &base) -> int {
        cudaStream_t s = ctx->copy_stream[slot];
        const uint64_t k0 = plan[c].k0, k1 = plan[c].k1;
        const uint64_t abs_base = offsets[k0] & ~511ull;
        KMPB_CUDA(cudaMemcpyAsync(ctx->d_stage_bytes[slot], bytes + abs_base, offsets[k1] - abs_base, cudaMemcpyHostToDevice, s));
        KMPB_CUDA(cudaMemcpyAsync(ctx->d_stage_off[slot], offsets + k0, (k1 - k0 + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, s));
        b = kmpb_batch{ctx->d_stage_bytes[slot], abs_base, ctx->d_stage_off[slot], k1 - k0, offsets[k0], offsets[k1]};
        base = k0;
        return KMPB_OK;
    };
    return find_chunks(ctx, plan.size(), max_bytes / 256, stage, out, capacity, n_found);
}

int kmpb_find_pcap(kmpb_ctx *ctx, const kmpb_pcap *pc, uint64_t first, uint64_t count, kmpb_match *out, uint64_t capacity,
                   uint64_t *n_found)
{
    if (pc == nullptr) return kmpb_fail(KMPB_EINVAL, "NULL argument");
    int rc = find_args(ctx, out, capacity, n_found);
    if (rc) return rc;
    *n_found = 0;
    if (ctx->host.n_pat == 0) return KMPB_OK;
    const uint64_t total = kmpb_pcap_packets(pc);
    if (first > total || count > total - first) return kmpb_fail(KMPB_EINVAL, "packet range outside the file");
    if (count == 0) return KMPB_OK;
    if ((rc = check_pcap_lengths(pc, first, count))) return rc;
    if ((rc = use_device(ctx))) return rc;
    const uint64_t chunk_bytes = chunk_bytes_setting();
    const uint64_t max_pkts = 1ull << 22, last = first + count;
    std::vector<uint64_t> starts; // first packet of every chunk, then `last`
    uint64_t max_bytes = 0, max_n = 0;
    for (uint64_t k0 = first; k0 < last;) {
        uint64_t nb = 0;
        const uint64_t k1 = kmpb_pcap_chunk_end(pc, k0, last, chunk_bytes, max_pkts, &nb);
        starts.push_back(k0);
        max_bytes = std::max(max_bytes, nb);
        max_n = std::max(max_n, k1 - k0);
        k0 = k1;
    }
    starts.push_back(last);
    if ((rc = ensure_staging(ctx, max_bytes, max_n))) return rc;
    if ((rc = ensure_host_staging(ctx, max_bytes, max_n))) return rc;
    if ((rc = kmpb_union_scratch(ctx, max_bytes))) return rc;
    // (a slot's pinned buffers are free again: its previous chunk has been finished, which waited for its stream)
    auto stage = [&](uint64_t c, int slot, kmpb_batch &b, uint64_t &base) -> int {
        cudaStream_t s = ctx->copy_stream[slot];
        const uint64_t k0 = starts[c], k1 = starts[c + 1];
        kmpb_pcap_pack(pc, k0, k1 - k0, ctx->h_stage_bytes[slot], ctx->h_stage_off[slot]);
        const uint64_t nbytes = ctx->h_stage_off[slot][k1 - k0];
        memset(ctx->h_stage_bytes[slot] + nbytes, 0, 64);
        KMPB_CUDA(cudaMemcpyAsync(ctx->d_stage_bytes[slot], ctx->h_stage_bytes[slot], nbytes + 64, cudaMemcpyHostToDevice, s));
        KMPB_CUDA(cudaMemcpyAsync(ctx->d_stage_off[slot], ctx->h_stage_off[slot], (k1 - k0 + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, s));
        b = kmpb_batch{ctx->d_stage_bytes[slot], 0, ctx->d_stage_off[slot], k1 - k0, 0, nbytes};
        base = k0;
        return KMPB_OK;
    };
    return find_chunks(ctx, starts.size() - 1, max_bytes / 256, stage, out, capacity, n_found);
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
    cudaStream_t s = ctx->copy_stream[slot];
    ctx->h_stage_off[slot][st->n] = st->bytes;
    memset(ctx->h_stage_bytes[slot] + st->bytes, 0, 64);
    KMPB_CUDA(cudaMemcpyAsync(ctx->d_stage_bytes[slot], ctx->h_stage_bytes[slot], st->bytes + 64, cudaMemcpyHostToDevice, s));
    KMPB_CUDA(cudaMemcpyAsync(ctx->d_stage_off[slot], ctx->h_stage_off[slot], (st->n + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, s));
    KMPB_CUDA(cudaEventRecord(ctx->ev_h2d[slot], s));
    kmpb_batch b{ctx->d_stage_bytes[slot], 0, ctx->d_stage_off[slot], st->n, 0, st->bytes};
    int rc = run_engine(ctx, b, slot, s); // accumulates into the slot's distinct-pattern counters
    if (rc) return rc;
    st->batches++;
    st->slot = (slot + 1) % KMPB_COPY_STREAMS;
    st->n = st->bytes = 0;
    if (st->batches >= (uint64_t)KMPB_COPY_STREAMS) KMPB_CUDA(cudaEventSynchronize(ctx->ev_h2d[st->slot])); // its last copy has left it
    return KMPB_OK;
}

int kmpb_stream_open(kmpb_ctx *ctx, int proto, uint64_t batch_bytes, kmpb_stream **out)
{
    if (ctx == nullptr || out == nullptr) return kmpb_fail(KMPB_EINVAL, "NULL argument");
    *out = nullptr;
    if (!ctx->have_tables) return kmpb_fail(KMPB_ESTATE, "stream before kmpb_set_patterns");
    if (proto != KMPB_PROTO_UDP && proto != KMPB_PROTO_TCP) return kmpb_fail(KMPB_EINVAL, "unknown protocol %d", proto);
    int rc = use_device(ctx);
    if (rc) return rc;
    if (batch_bytes == 0) batch_bytes = 8ull << 20;
    if (batch_bytes < 65536) batch_bytes = 65536; // a frame's payload is at most 65535 - headers bytes long... jumbo included
    const uint64_t max_pkts = 1ull << 20;
    if ((rc = ensure_staging(ctx, batch_bytes, max_pkts))) return rc;
    if ((rc = ensure_host_staging(ctx, batch_bytes, max_pkts))) return rc;
    if ((rc = kmpb_union_scratch(ctx, batch_bytes))) return rc;
    const uint32_t nu = ctx->host.n_uniq;
    KMPB_CUDA(cudaEventRecord(ctx->ev[0], ctx->stream));
    KMPB_CUDA(cudaMemsetAsync(ctx->d_uniq_counts, 0, (size_t)KMPB_COPY_STREAMS * (nu ? nu : 1) * sizeof(uint64_t), ctx->stream));
    KMPB_CUDA(cudaStreamSynchronize(ctx->stream));
    kmpb_stream *st = new (std::nothrow) kmpb_stream();
    if (st == nullptr) return kmpb_fail(KMPB_ENOMEM, "out of memory");
    st->ctx = ctx;
    st->extract = proto == KMPB_PROTO_TCP ? kmpb_extract_tcp : kmpb_extract_udp;
    st->batch_bytes = batch_bytes;
    st->max_pkts = max_pkts;
    st->slot = 0;
    st->n = st->bytes = st->batches = st->frames = st->packets = 0;
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
    ctx->h_stage_off[st->slot][st->n] = st->bytes;
    memcpy(ctx->h_stage_bytes[st->slot] + st->bytes, frame + off, len);
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
