// select.cu -- which packets match: the mark kernel's start-position bitmap turned into one verdict per packet, and the
// indices of the selected packets.
//
// The mark kernel (union_kernel.cu, kmpb_union_mark_kernel) counts like the count kernel and, for every match it
// verifies, sets the bit of the match's first byte in a bitmap of the batch: bit p & 31 of word (p >> 5) - (first_byte
// >> 5).  The verifier does not know a candidate's packet (a candidate-ring slot holds its text, position and room
// only), and a bitmap needs no slot reservation and no capacity: it is 1/8 of the batch's span, known before the launch.
// Two small passes follow:
//   - verdict: a thread reads four words, and for each set bit finds the packet that holds that byte (an interpolation
//     guess for the first, a search up from the last one found for the others), sets its flag, clears the word's bits
//     up to that packet's end and repeats -- so a word whose bits span many small packets costs one search
//     per packet, not per bit.  It zeroes every non-zero word it read: the bitmap is all zero again after the pass, with
//     no memset per call.
//   - compaction (device form only): the ascending indices of the flagged (or, inverted, unflagged) packets, CUB's
//     DeviceSelect over the packet indices.
#include <cub/device/device_select.cuh>
#include <thrust/iterator/counting_iterator.h>
#include <thrust/iterator/discard_iterator.h>

#include "kmpb_device.cuh"

constexpr int VERDICT_THREADS = 256;
constexpr uint64_t VERDICT_TILE = 4 * VERDICT_THREADS; // words per block: one 16-byte load per thread

// the last k in [lo, hi) with offsets[k] <= pos, given offsets[lo] <= pos or lo == 0
__device__ __forceinline__ uint64_t packet_in(const uint64_t *__restrict__ offsets, uint64_t lo, uint64_t hi, uint64_t pos)
{
    while (hi - lo > 1) {
        const uint64_t mid = lo + (hi - lo) / 2;
        if (offsets[mid] <= pos) lo = mid; else hi = mid;
    }
    return lo;
}

// the last k < n with offsets[k] <= pos, given offsets[k0] <= pos: doubling steps up from k0, then bisection -- a few
// dependent loads when the answer is near k0, as it is for the bits of one word after the first
__device__ __forceinline__ uint64_t packet_from(const uint64_t *__restrict__ offsets, uint64_t k0, uint64_t n, uint64_t pos)
{
    uint64_t lo = k0, hi = n; // offsets[lo] <= pos < offsets[hi] (hi = n: past the end)
    for (uint64_t step = 1; lo + step < n; step *= 2) {
        if (offsets[lo + step] > pos) { hi = lo + step; break; }
        lo += step;
    }
    return packet_in(offsets, lo, hi, pos);
}

// the last k < n with offsets[k] <= pos, for offsets[0] <= pos < offsets[n]: a guess by the mean packet size (exact for
// equal-sized packets), a bracket by doubling steps around it, then bisection -- a few dependent loads where a plain
// binary search over millions of packets takes twenty-odd
__device__ __forceinline__ uint64_t packet_near(const uint64_t *__restrict__ offsets, uint64_t n, uint64_t pos)
{
    const uint64_t first = offsets[0], total = offsets[n] - first;
    uint64_t g = (uint64_t)((double)(pos - first) / (double)total * (double)n);
    g = g >= n ? n - 1 : g;
    if (offsets[g] <= pos) return packet_from(offsets, g, n, pos);
    uint64_t hi = g, lo = 0;
    for (uint64_t step = 1; step <= hi; step *= 2) {
        if (offsets[hi - step] <= pos) { lo = hi - step; break; }
        hi -= step;
    }
    return packet_in(offsets, lo, hi, pos);
}

// words[n_words] (n_words a multiple of 4): bit j of word w stands for absolute byte base + 32 w + j (base a multiple of
// 32).  flags[k] = 1 for every packet k that holds a set bit; every word read is left zero.  A thread reads four words;
// one whose words are all zero (most of them) is done at once -- no block-wide step waits for anything.  For its first
// set bit a thread guesses the packet by interpolation; every later bit's packet lies at or after the last one found.
__global__ void __launch_bounds__(VERDICT_THREADS) kmpb_verdict_kernel(uint32_t *__restrict__ words, uint64_t n_words, uint64_t base,
                                                                       const uint64_t *__restrict__ offsets, uint64_t n_packets,
                                                                       uint8_t *__restrict__ flags)
{
    const uint64_t w = 4 * ((uint64_t)blockIdx.x * VERDICT_THREADS + threadIdx.x);
    if (w >= n_words) return;
    uint4 *const at = reinterpret_cast<uint4 *>(words + w);
    const uint4 v = *at;
    if ((v.x | v.y | v.z | v.w) == 0) return;
    *at = make_uint4(0, 0, 0, 0);
    const uint32_t vs[4] = {v.x, v.y, v.z, v.w};
    bool found = false;
    uint64_t k = 0;
#pragma unroll
    for (int j = 0; j < 4; j++) {
        uint32_t x = vs[j];
        const uint64_t wb = base + 32 * (w + j);
        while (x) { // a set bit lies in a non-empty packet of the batch: the last k with offsets[k] <= its byte
            const uint64_t pos = wb + (uint32_t)(__ffs(x) - 1);
            k = found ? packet_from(offsets, k, n_packets, pos) : packet_near(offsets, n_packets, pos);
            found = true;
            flags[k] = 1;
            const uint64_t e = offsets[k + 1];
            if (e >= wb + 32) break;
            x &= ~((1u << (uint32_t)(e - wb)) - 1u); // the bits of packet k (e - wb is 1..31)
            k++;                                     // offsets[k] = e <= every bit left
        }
    }
}

namespace {

// selected: the flag is set (or, inverted, clear)
struct flag_is {
    const uint8_t *flags;
    bool want;
    __device__ __forceinline__ bool operator()(uint64_t i) const { return (flags[i] != 0) == want; }
};

} // namespace

uint64_t kmpb_mark_words(const kmpb_batch &b)
{
    const uint64_t bits = b.end_byte - (b.first_byte & ~31ull);
    return ((bits + 31) / 32 + 3) & ~3ull;
}

int kmpb_ensure_mark(kmpb_ctx *ctx, int slot, uint64_t words, cudaStream_t stream)
{
    words = (words + 3) & ~3ull;
    kmpb_scratch<uint32_t> &mark = ctx->d_mark[slot];
    if (words > mark.cap || !mark.p) {
        if (int rc = mark.reserve(words > 4 ? words : 4)) return rc;
        ctx->mark_dirty[slot] = true; // zeroed below on `stream`, ahead of the mark kernel that runs there
    }
    // (cudaMemset would run on the legacy default stream, which the context's non-blocking streams do not wait for: the
    // zeros could land after the mark kernel's bits.)  After every device-form call issued so far: slot 0's bitmap is
    // theirs as well.
    if (ctx->mark_dirty[slot]) {
        KMPB_CUDA(cudaStreamWaitEvent(stream, ctx->ev_dev, 0));
        KMPB_CUDA(cudaMemsetAsync(mark.p, 0, mark.cap * sizeof(uint32_t), stream));
        ctx->mark_dirty[slot] = false;
    }
    return KMPB_OK;
}

int kmpb_select_match(kmpb_ctx *ctx, const kmpb_batch &b, int slot, uint8_t *d_flags, cudaStream_t stream,
                      const kmpb_fused_out &out)
{
    if (b.n_packets) KMPB_CUDA(cudaMemsetAsync(d_flags, 0, b.n_packets, stream));
    const kmpb_tables &h = ctx->host;
    if (h.n_uniq == 0 || b.n_packets == 0 || b.end_byte == b.first_byte) return KMPB_OK;
    const uint64_t words = kmpb_mark_words(b);
    int rc = kmpb_ensure_mark(ctx, slot, words, stream);
    if (rc) return rc;
    ctx->mark_dirty[slot] = true; // until the verdict pass is on its way
    if ((rc = kmpb_launch_union(ctx, b, slot, ctx->d_uniq_counts + (size_t)slot * h.n_uniq, stream, out, nullptr, ctx->d_mark[slot].p)))
        return rc;
    const uint64_t blocks = (words + VERDICT_TILE - 1) / VERDICT_TILE;
    kmpb_verdict_kernel<<<(unsigned)blocks, VERDICT_THREADS, 0, stream>>>(ctx->d_mark[slot].p, words, b.first_byte & ~31ull,
                                                                         b.d_offsets, b.n_packets, d_flags);
    ctx->launches++;
    KMPB_CUDA(cudaGetLastError());
    if (ctx->profile) KMPB_CUDA(cudaEventRecord(ctx->ev_kernel[1], stream)); // the bracket covers mark + verdict
    ctx->mark_dirty[slot] = false;
    return KMPB_OK;
}

int kmpb_select_compact(kmpb_ctx *ctx, const uint8_t *d_flags, uint64_t n_packets, bool invert, uint64_t *d_index,
                        uint64_t *d_n_selected, cudaStream_t stream)
{
    if (n_packets == 0) {
        KMPB_CUDA(cudaMemsetAsync(d_n_selected, 0, sizeof(uint64_t), stream));
        return KMPB_OK;
    }
    const thrust::counting_iterator<uint64_t> in(0);
    const flag_is pred{d_flags, !invert};
    const int64_t n = (int64_t)n_packets;
    size_t need = 0;
    if (d_index) KMPB_CUDA(cub::DeviceSelect::If(nullptr, need, in, d_index, d_n_selected, n, pred, stream));
    else KMPB_CUDA(cub::DeviceSelect::If(nullptr, need, in, thrust::discard_iterator<>(), d_n_selected, n, pred, stream));
    if (int rc = ctx->d_select_temp.reserve(need)) return rc;
    size_t temp = ctx->d_select_temp.cap;
    if (d_index) KMPB_CUDA(cub::DeviceSelect::If(ctx->d_select_temp.p, temp, in, d_index, d_n_selected, n, pred, stream));
    else KMPB_CUDA(cub::DeviceSelect::If(ctx->d_select_temp.p, temp, in, thrust::discard_iterator<>(), d_n_selected, n, pred, stream));
    ctx->launches += 2;
    return KMPB_OK;
}
