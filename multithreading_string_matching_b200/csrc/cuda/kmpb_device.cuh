// kmpb_device.cuh -- context layout and launch entry points shared by the .cu files of libkmpb200.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "../host/kmpb_internal.h"

#define KMPB_CUDA(call)                                                                          \
    do {                                                                                         \
        cudaError_t e_ = (call);                                                                 \
        if (e_ != cudaSuccess)                                                                   \
            return kmpb_fail(KMPB_ECUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), \
                             __FILE__, __LINE__);                                                \
    } while (0)

constexpr int KMPB_COPY_STREAMS = 4;          // stream slots of the chunk pipeline of the host and savefile forms
constexpr uint32_t KMPB_SMEM_COUNTS_MAX = 4096; // distinct patterns counted in shared memory; above: global atomics

// Per-context scratch that grows on demand: p holds cap elements of T, in device memory (pinned host memory when
// PINNED); cap is 0 exactly when p is null.  reserve(n) keeps a buffer that holds n elements already.  Otherwise it
// synchronises the device (a call in flight may still use the old buffer), frees the old buffer and allocates n
// elements, whose contents are undefined.  With `zero` (device buffers) they are zero before it returns: the zeros go
// out on the legacy default stream, which the context's non-blocking streams do not wait for, so it waits for them
// itself.  A failure leaves the buffer null with capacity 0.
template <class T, bool PINNED = false>
struct kmpb_scratch {
    T *p = nullptr;
    uint64_t cap = 0;

    int reserve(uint64_t n, bool zero = false)
    {
        if (p && n <= cap) return KMPB_OK;
        if (p) {
            KMPB_CUDA(cudaDeviceSynchronize());
            release();
        }
        const size_t bytes = n * sizeof(T);
        void *q = nullptr;
        cudaError_t e = PINNED ? cudaHostAlloc(&q, bytes, cudaHostAllocDefault) : cudaMalloc(&q, bytes);
        if (e != cudaSuccess)
            return kmpb_fail(KMPB_ECUDA, "allocating %zu bytes of %s scratch failed: %s", bytes, PINNED ? "pinned" : "device",
                             cudaGetErrorString(e));
        p = static_cast<T *>(q);
        cap = n;
        if (zero && ((e = cudaMemsetAsync(p, 0, bytes, 0)) != cudaSuccess || (e = cudaStreamSynchronize(0)) != cudaSuccess)) {
            release();
            return kmpb_fail(KMPB_ECUDA, "zeroing %zu bytes of scratch failed: %s", bytes, cudaGetErrorString(e));
        }
        return KMPB_OK;
    }

    void release()
    {
        if (PINNED) cudaFreeHost(p);
        else cudaFree(p);
        p = nullptr;
        cap = 0;
    }
};

// Device-resident tables of one pattern set (device pointers).
struct kmpb_device_tables {
    uint32_t n_pat = 0, n_uniq = 0, n_class = 0, n_state = 0, max_len = 0, min_len = 0;
    // distinct patterns
    uint8_t *uniq_blob = nullptr;   // [sum len]
    uint32_t *uniq_off = nullptr;   // [n_uniq+1]
    uint32_t *uniq_len = nullptr;   // [n_uniq]
    uint8_t *uniq_flags = nullptr;  // [n_uniq] KMPB_PAT_NOCASE or 0
    uint32_t *pat_to_uniq = nullptr; // [n_pat]
    // per-pattern engine: failure tables and byte-indexed KMP DFAs, both built on the device
    int32_t *pi = nullptr;          // [sum len], pattern u at uniq_off[u]
    uint8_t *perpat_dfa = nullptr;  // pattern u: uniq_len[u] rows of 256 entries at 256*uniq_off[u]
    // union engine
    uint32_t *vtab = nullptr;       // [vtab_words] start-anchored verification tables (automaton.c)
    uint32_t *filter = nullptr;     // [256]
    uint32_t *gate = nullptr;       // [host.gate_words] prefix gate (automaton.c build_gate), null when there is none
    uint32_t *uniq_first = nullptr; // [n_uniq] lowest file-order index of each distinct pattern (the find records' pattern)
    // window kernel: the windowed patterns' probe tables and windows (automaton.c), null when the set has none
    uint32_t *wvtab = nullptr;      // [host.wvtab_words]
    uint32_t *uniq_lo = nullptr, *uniq_hi = nullptr; // [n_uniq - host.n_union]
};

struct kmpb_ctx {
    int device = 0;
    int sm_count = 0;
    int engine = KMPB_ENGINE_AUTO;
    size_t smem_optin = 0;
    cudaStream_t stream = nullptr;                      // default stream of the context
    cudaStream_t copy_stream[KMPB_COPY_STREAMS] = {};   // copies + kernels of one stream slot (chunk pipeline, frame stream)
    cudaEvent_t ev[4] = {};
    cudaEvent_t ev_kernel[2] = {};                      // around the dominant kernel when profile is on
    cudaEvent_t ev_dev = nullptr;                       // after the last device-form call's work, on its stream
    int open_streams = 0;                               // kmpb_stream_open without kmpb_stream_close yet
    bool profile = false;
    kmpb_tables host = {};
    bool have_tables = false;
    kmpb_device_tables dev;
    uint64_t *d_uniq_counts = nullptr;   // [n_uniq] per-launch accumulators (per stream slot), with the tables
    uint64_t *d_counts = nullptr;        // [n_pat] counts of the last finished chunked call (kmpb_device_counts)
    // scratch, grown on demand
    kmpb_scratch<uint32_t> d_work;       // work counters, 4 words per stream slot (word 1: error flags)
    kmpb_scratch<uint32_t> d_items;      // item -> first packet table, cap / KMPB_COPY_STREAMS entries per stream slot
    // the staging slots of the host and savefile forms and the frame stream, and their pinned twins, into which
    // savefile chunks and pushed frames are packed first
    kmpb_scratch<uint8_t> d_stage_bytes[KMPB_COPY_STREAMS];
    kmpb_scratch<uint64_t> d_stage_off[KMPB_COPY_STREAMS];
    kmpb_scratch<uint8_t, true> h_stage_bytes[KMPB_COPY_STREAMS];
    kmpb_scratch<uint64_t, true> h_stage_off[KMPB_COPY_STREAMS];
    cudaEvent_t ev_h2d[KMPB_COPY_STREAMS] = {};
    // find: record buffers and found counters of the chunked forms (per stream slot), the sort's keys and CUB scratch
    kmpb_scratch<kmpb_match> d_find_rec[KMPB_COPY_STREAMS];
    kmpb_scratch<unsigned long long> d_find_found; // [KMPB_COPY_STREAMS]
    kmpb_scratch<uint64_t> d_sort_keys[2];
    kmpb_scratch<uint8_t> d_sort_temp;
    // select: the start-position bitmaps (per stream slot: one bit per payload byte, all zero between calls), the
    // verdicts of the chunked forms (per slot, device and pinned host), the compaction's CUB scratch
    kmpb_scratch<uint32_t> d_mark[KMPB_COPY_STREAMS];
    bool mark_dirty[KMPB_COPY_STREAMS] = {};   // a call failed after its mark kernel: the bitmap may hold bits
    kmpb_scratch<uint8_t> d_sel_flags[KMPB_COPY_STREAMS];
    kmpb_scratch<uint8_t, true> h_sel_flags[KMPB_COPY_STREAMS];
    kmpb_scratch<uint8_t> d_select_temp;
    bool attr_union_set = false, attr_perpat_set = false; // per-device function attributes
    uint64_t launches = 0;
    double last_ms[2] = {0, 0};
};

// One batch on the device.  d_bytes[0] is absolute byte `abs_base` of the CSR byte space (a multiple
// of 512); offsets are absolute.  All launches go to `stream`; slot selects the scratch set.
struct kmpb_batch {
    const uint8_t *d_bytes;
    uint64_t abs_base;
    const uint64_t *d_offsets; // [n_packets+1]
    uint64_t n_packets;
    uint64_t first_byte, end_byte; // offsets[0], offsets[n_packets] (host copies)
};

// Where the union kernel's last block adds the per-pattern counts (file order) itself: up to 8 count
// vectors, this GPU's and/or peers' mapped over NVLink.  n = 0: the caller expands the counts afterwards.
constexpr int KMPB_MAX_OUT = 8;
struct kmpb_fused_out {
    unsigned long long *vec[KMPB_MAX_OUT] = {};
    uint32_t n = 0;
};

// Where the find kernel writes its records: rec[capacity] of {absolute position, 0, distinct id} (find.cu turns them
// into kmpb_match), *found counts every match, also those past the capacity.
struct kmpb_find_out {
    kmpb_match *rec = nullptr;
    uint64_t capacity = 0;
    unsigned long long *found = nullptr;
};

// tables.cu
int kmpb_upload_tables(kmpb_ctx *ctx);
void kmpb_release_tables(kmpb_ctx *ctx);
// perpat_kernel.cu
int kmpb_launch_perpat(kmpb_ctx *ctx, const kmpb_batch &b, uint64_t *d_uniq_counts, cudaStream_t stream);
// union_kernel.cu
// mark (select.cu): the start-position bitmap of the batch, word 0 holding byte first_byte (find must be null)
int kmpb_launch_union(kmpb_ctx *ctx, const kmpb_batch &b, int slot, uint64_t *d_uniq_counts, cudaStream_t stream,
                      const kmpb_fused_out &out = kmpb_fused_out(), const kmpb_find_out *find = nullptr,
                      uint32_t *mark = nullptr);
int kmpb_union_scratch(kmpb_ctx *ctx, uint64_t max_batch_bytes);
// window.cu: the windowed patterns of a batch (launched by kmpb_launch_union alone, before its own kernels): counts into
// d_uniq_counts, records into *find or bits into the biased bitmap mark_biased (as the union kernel's), and the
// file-order counts added to out when out.n > 0 (the caller passes that only when the union kernel does not run)
int kmpb_launch_window(kmpb_ctx *ctx, const kmpb_batch &b, uint32_t *d_work, uint64_t *d_uniq_counts, cudaStream_t stream,
                       const kmpb_fused_out &out, const kmpb_find_out *find, uint32_t *mark_biased);
// find.cu: the find kernel into d_rec[capacity] (*d_found = every match of the batch), then the records turned into
// kmpb_match (packet index + packet_base), sorted or not
int kmpb_find_match(kmpb_ctx *ctx, const kmpb_batch &b, int slot, kmpb_match *d_rec, uint64_t capacity, unsigned long long *d_found,
                    cudaStream_t stream);
int kmpb_find_finish(kmpb_ctx *ctx, const kmpb_batch &b, uint64_t packet_base, kmpb_match *d_rec, uint64_t capacity,
                     const unsigned long long *d_found, bool sorted, cudaStream_t stream);
// select.cu: the words of a batch's start-position bitmap; the bitmap of a stream slot at least that long (zeroed when
// allocated and when a failed call left it dirty, on `stream`); mark kernel + verdict into d_flags[n_packets] (zeroed
// first), the counts added to the slot's distinct-pattern counters (and to out when out.n > 0); the ascending indices
// of the packets whose flag is (invert ? 0 : 1) into d_index (may be null) and their number into *d_n_selected
uint64_t kmpb_mark_words(const kmpb_batch &b);
int kmpb_ensure_mark(kmpb_ctx *ctx, int slot, uint64_t words, cudaStream_t stream);
int kmpb_select_match(kmpb_ctx *ctx, const kmpb_batch &b, int slot, uint8_t *d_flags, cudaStream_t stream,
                      const kmpb_fused_out &out = kmpb_fused_out());
int kmpb_select_compact(kmpb_ctx *ctx, const uint8_t *d_flags, uint64_t n_packets, bool invert, uint64_t *d_index,
                        uint64_t *d_n_selected, cudaStream_t stream);
// api.cu
int kmpb_launch_expand(kmpb_ctx *ctx, const uint64_t *d_uniq_counts, uint64_t *d_counts, cudaStream_t stream);
