// find.cu -- where the patterns occur: the find kernel's records turned into kmpb_match, optionally sorted.
//
// The find kernel (union_kernel.cu, kmpb_union_find_kernel) writes one record per match, {absolute position, 0,
// distinct pattern id}, in whatever order its warps verify candidates.  What it does not know cheaply is the packet:
// the resolve step keeps the packet bounds of a candidate, not its index.  So a small pass follows:
//   - locate: packet = the last k with offsets[k] <= position (a binary search in the batch's offsets; a matched byte
//     lies in a non-empty packet, so empty packets never win), offset = position - offsets[k], pattern = the lowest
//     file-order index of the distinct id (uniq_first, built with the tables);
//   - sorted: every record becomes one 64-bit key, (position - first_byte) << pbits | pattern; the keys are radix-sorted
//     (CUB, only the bits in use) and the locate step reads the sorted keys.  Ordering by position orders by (packet,
//     offset), because packets are consecutive byte ranges of the batch.
#include <cub/device/device_radix_sort.cuh>

#include "kmpb_device.cuh"

constexpr int FIND_THREADS = 256;

__device__ __forceinline__ uint64_t n_written(const unsigned long long *found, uint64_t capacity)
{
    const uint64_t n = *found;
    return n < capacity ? n : capacity;
}

// the packet that holds absolute byte `pos`: the last k < n_packets with offsets[k] <= pos
__device__ __forceinline__ uint64_t packet_of(const uint64_t *__restrict__ offsets, uint64_t n_packets, uint64_t pos)
{
    uint64_t lo = 0, hi = n_packets;
    while (hi - lo > 1) {
        const uint64_t mid = lo + (hi - lo) / 2;
        if (offsets[mid] <= pos) lo = mid; else hi = mid;
    }
    return lo;
}

__global__ void kmpb_locate_kernel(kmpb_match *__restrict__ rec, uint64_t capacity, const unsigned long long *__restrict__ found,
                                   const uint64_t *__restrict__ offsets, uint64_t n_packets, const uint32_t *__restrict__ uniq_first,
                                   uint64_t packet_base)
{
    const uint64_t n = n_written(found, capacity);
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        const kmpb_match r = rec[i];
        const uint64_t k = packet_of(offsets, n_packets, r.packet);
        rec[i] = kmpb_match{packet_base + k, (uint32_t)(r.packet - offsets[k]), uniq_first[r.pattern]};
    }
}

// the sort keys of the records; slots [n, capacity) get the largest key, so that they sort behind every record
__global__ void kmpb_find_keys_kernel(const kmpb_match *__restrict__ rec, uint64_t capacity, const unsigned long long *__restrict__ found,
                                      uint64_t first_byte, uint32_t pbits, const uint32_t *__restrict__ uniq_first,
                                      uint64_t *__restrict__ keys)
{
    const uint64_t n = n_written(found, capacity);
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < capacity; i += (uint64_t)gridDim.x * blockDim.x) {
        uint64_t key = ~0ull;
        if (i < n) {
            const kmpb_match r = rec[i];
            key = ((r.packet - first_byte) << pbits) | uniq_first[r.pattern];
        }
        keys[i] = key;
    }
}

__global__ void kmpb_locate_keys_kernel(const uint64_t *__restrict__ keys, uint64_t capacity, const unsigned long long *__restrict__ found,
                                        uint64_t first_byte, uint32_t pbits, const uint64_t *__restrict__ offsets, uint64_t n_packets,
                                        uint64_t packet_base, kmpb_match *__restrict__ out)
{
    const uint64_t n = n_written(found, capacity);
    const uint64_t pmask = (1ull << pbits) - 1ull;
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t key = keys[i];
        const uint64_t pos = first_byte + (key >> pbits);
        const uint64_t k = packet_of(offsets, n_packets, pos);
        out[i] = kmpb_match{packet_base + k, (uint32_t)(pos - offsets[k]), (uint32_t)(key & pmask)};
    }
}

namespace {

uint32_t bits_for(uint64_t max_value) { return max_value ? 64u - (uint32_t)__builtin_clzll(max_value) : 0u; }

int grid_for(const kmpb_ctx *ctx, uint64_t n)
{
    const uint64_t blocks = (n + FIND_THREADS - 1) / FIND_THREADS, most = 8ull * (uint64_t)ctx->sm_count;
    return (int)(blocks < 1 ? 1 : blocks < most ? blocks : most);
}

// the sort's key buffers (two of `items` keys) and CUB's temporary storage, grown on demand
int ensure_sort_scratch(kmpb_ctx *ctx, uint64_t items, uint32_t end_bit, cudaStream_t stream)
{
    int rc;
    if ((rc = ctx->d_sort_keys[0].reserve(items)) || (rc = ctx->d_sort_keys[1].reserve(items))) return rc;
    cub::DoubleBuffer<uint64_t> db(ctx->d_sort_keys[0].p, ctx->d_sort_keys[1].p);
    size_t need = 0;
    KMPB_CUDA(cub::DeviceRadixSort::SortKeys(nullptr, need, db, (int)items, 0, (int)end_bit, stream));
    return ctx->d_sort_temp.reserve(need);
}

} // namespace

int kmpb_find_match(kmpb_ctx *ctx, const kmpb_batch &b, int slot, kmpb_match *d_rec, uint64_t capacity, unsigned long long *d_found,
                    cudaStream_t stream)
{
    const kmpb_tables &h = ctx->host;
    KMPB_CUDA(cudaMemsetAsync(d_found, 0, sizeof(unsigned long long), stream));
    if (h.n_uniq == 0 || b.n_packets == 0 || b.end_byte == b.first_byte) return KMPB_OK;
    kmpb_find_out fo;
    fo.rec = d_rec;
    fo.capacity = capacity;
    fo.found = d_found;
    return kmpb_launch_union(ctx, b, slot, ctx->d_uniq_counts + (size_t)slot * h.n_uniq, stream, kmpb_fused_out(), &fo);
}

int kmpb_find_finish(kmpb_ctx *ctx, const kmpb_batch &b, uint64_t packet_base, kmpb_match *d_rec, uint64_t capacity,
                     const unsigned long long *d_found, bool sorted, cudaStream_t stream)
{
    const kmpb_tables &h = ctx->host;
    if (capacity == 0 || h.n_uniq == 0 || b.n_packets == 0 || b.end_byte == b.first_byte) return KMPB_OK;
    if (!sorted) {
        kmpb_locate_kernel<<<grid_for(ctx, capacity), FIND_THREADS, 0, stream>>>(d_rec, capacity, d_found, b.d_offsets, b.n_packets,
                                                                                 ctx->dev.uniq_first, packet_base);
        ctx->launches++;
        KMPB_CUDA(cudaGetLastError());
        return KMPB_OK;
    }
    const uint32_t pbits = bits_for(h.n_pat - 1), end_bit = bits_for(b.end_byte - b.first_byte - 1) + pbits;
    if (end_bit > 64) return kmpb_fail(KMPB_ELIMIT, "sorted records: bits of the batch's span + bits of the pattern count exceed 64");
    if (capacity > (uint64_t)INT32_MAX) return kmpb_fail(KMPB_ELIMIT, "sorted records: more than 2^31-1 records in one sort");
    const int bits = end_bit ? (int)end_bit : 1;
    int rc = ensure_sort_scratch(ctx, capacity, (uint32_t)bits, stream);
    if (rc) return rc;
    kmpb_find_keys_kernel<<<grid_for(ctx, capacity), FIND_THREADS, 0, stream>>>(d_rec, capacity, d_found, b.first_byte, pbits,
                                                                                ctx->dev.uniq_first, ctx->d_sort_keys[0].p);
    KMPB_CUDA(cudaGetLastError());
    cub::DoubleBuffer<uint64_t> db(ctx->d_sort_keys[0].p, ctx->d_sort_keys[1].p);
    size_t temp = ctx->d_sort_temp.cap;
    KMPB_CUDA(cub::DeviceRadixSort::SortKeys(ctx->d_sort_temp.p, temp, db, (int)capacity, 0, bits, stream));
    kmpb_locate_keys_kernel<<<grid_for(ctx, capacity), FIND_THREADS, 0, stream>>>(db.Current(), capacity, d_found, b.first_byte, pbits,
                                                                                  b.d_offsets, b.n_packets, packet_base, d_rec);
    ctx->launches += 3;
    KMPB_CUDA(cudaGetLastError());
    return KMPB_OK;
}
