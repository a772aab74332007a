// window.cu -- the window kernel: the patterns with a position window [lo, hi] (kmpb_set_patterns_win).
//
// The union kernel cannot test a window: its candidates carry an absolute position, not a packet and an offset in it.
// So the windowed patterns are matched in a pass of their own, launched by kmpb_launch_union before its own kernels on
// the same stream, and it reads only the head of every packet: a pattern of length m whose window ends at hi can only
// touch the packet's first hi + m bytes, so bytes [0, min(len, W)) with W = max(hi + m) are all it needs.
//
// One warp takes one packet at a time.  It walks the head in tiles of WN_TILE start offsets: the tile's bytes and the
// WN_LOOK bytes after it (a match that starts in the tile ends inside them) go from global memory to the warp's buffer
// in shared memory by coalesced 16-byte loads; the same pass finds the first NUL byte among them.  The tiles come in
// order, so a NUL seen in a tile is the packet's first, and the walk stops once no start before it is left.  Each lane then
// tests 32 start offsets of the tile (four per buffer word, the words of the warp's lanes adjacent: no bank
// conflicts): a start whose first byte begins no windowed pattern (a 256-bit table) ends there, the others are looked
// up in the windowed patterns' probe tables (automaton.c build_verify_tables, the layout of the union kernel's tables)
// with the same masked compare.  A record that agrees is a match when the pattern ends inside the packet and before
// its first NUL and the start lies in the pattern's own window.
//
// A hit does what the union kernel's does: count (64-bit shared-memory counters, one atomic per block and pattern at
// the end), find (a record {absolute position, 0, distinct id} in a slot reserved from the same found counter) or mark
// (the start bit in the select bitmap).  When every pattern of the set is windowed the union kernel does not run, and
// the last block of this one adds the file-order counts to the fused count vectors instead.
#include <cooperative_groups.h>

#include "kmpb_device.cuh"

constexpr int WN_THREADS = 256;
constexpr int WN_WARPS = WN_THREADS / 32;
constexpr int WN_BLOCKS_PER_SM = 4; // resident blocks an SM (up to 64 registers a thread), the grid's size
constexpr uint32_t WN_TILE = 1024;                    // start offsets per tile: 32 per lane
constexpr uint32_t WN_LOOK = 128;                     // bytes after the tile: a match that starts in it ends there
constexpr uint32_t WN_BUF_WORDS = (WN_TILE + WN_LOOK + 16 + 128) / 4; // + lead to the 16-byte boundary + slack for the
                                                                      // word reads past the last start
static_assert(WN_LOOK >= KMPB_MAX_PATTERN_LEN + 8, "the lookahead holds the longest pattern");

enum : int { WN_COUNT = 0, WN_FIND = 1, WN_MARK = 2 };

struct window_params {
    const uint8_t *bytes; // device pointer to absolute byte abs_base
    uint64_t abs_base;
    const uint64_t *offsets; // [n_packets+1], absolute
    uint64_t n_packets;
    const uint32_t *vtab;    // the windowed patterns' probe tables (global), vtab_words words
    uint32_t vtab_words, vtab_in_smem;
    uint32_t slots_a, shift_a, slots_b, shift_b, one, rec, blob; // its header words
    uint32_t nocase;         // the tables have the nocase layout
    const uint32_t *lo, *hi; // [n_win] window of distinct id u0 + w
    const uint8_t *uniq_blob, *uniq_flags; // the distinct patterns (one-byte runs: window_probe)
    const uint32_t *uniq_off, *uniq_len;
    uint32_t u0, n_win;
    uint32_t lo_min, hi_max, reach;
    uint32_t first[8];       // bytes a windowed pattern can start with
    unsigned long long *uniq_counts;
    uint32_t counts_in_smem;
    uint32_t *work;          // the slot's work words: [1] error flags, [3] blocks that have finished (expansion)
    // find: records and found counter; mark: the start-position bitmap, biased (as the union kernel's)
    kmpb_match *rec_out;
    uint64_t capacity;
    unsigned long long *found;
    uint32_t *mark;
    // expansion when the union kernel does not run: n_out count vectors
    const uint32_t *pat_to_uniq;
    uint32_t n_pat, n_out;
    unsigned long long *out[KMPB_MAX_OUT];
};

template <int OUT>
__device__ __forceinline__ void window_hit(const window_params &p, unsigned long long *s_counts, uint32_t u, uint64_t pos)
{
    if (s_counts) atomicAdd(s_counts + (u - p.u0), 1ull);
    else atomicAdd(p.uniq_counts + u, 1ull);
    if (OUT == WN_FIND) {
        namespace cg = cooperative_groups;
        const cg::coalesced_group g = cg::coalesced_threads();
        unsigned long long base = 0;
        if (g.thread_rank() == 0) base = atomicAdd(p.found, (unsigned long long)g.size());
        const uint64_t slot = g.shfl(base, 0) + g.thread_rank();
        if (slot < p.capacity)
            __stcs(reinterpret_cast<uint4 *>(p.rec_out) + slot, make_uint4((uint32_t)pos, (uint32_t)(pos >> 32), 0u, u));
    }
    if (OUT == WN_MARK) asm volatile("red.global.or.b32 [%0], %1;" ::"l"(p.mark + (pos >> 5)), "r"(1u << (uint32_t)(pos & 31u)) : "memory");
}

// 4 bytes of the warp's buffer from byte j on
__device__ __forceinline__ uint32_t buf_word(const uint32_t *buf, uint32_t j)
{
    return __funnelshift_r(buf[j >> 2], buf[(j >> 2) + 1], 8u * (j & 3u));
}

// The start at packet offset o (buffer byte j, first text bytes x0, x1), `room` = text bytes from o to the text's end
// (the packet's end or its first NUL, whichever comes first): every windowed pattern that starts there, fits the room
// and has o in its window.
template <int OUT>
__device__ __forceinline__ void window_probe(const window_params &p, const uint32_t *vt, unsigned long long *s_counts,
                                             const uint32_t *buf, uint32_t j, uint32_t x0, uint32_t x1, uint32_t o,
                                             uint32_t room, uint64_t pos)
{
    auto in_window = [&](uint32_t u) { return o >= __ldg(p.lo + (u - p.u0)) && o <= __ldg(p.hi + (u - p.u0)); };
    // One-byte patterns: the table holds the last id of the run of windowed patterns with that byte and flag (their ids
    // are consecutive, automaton.c cmp_distinct), which differ in their windows alone.
    auto one_byte = [&](uint32_t u) {
        if (u == 0xffffffffu) return;
        const uint8_t c = __ldg(p.uniq_blob + __ldg(p.uniq_off + u)), f = __ldg(p.uniq_flags + u);
        for (uint32_t v = u;; v--) {
            if (in_window(v)) window_hit<OUT>(p, s_counts, v, pos);
            if (v == p.u0 || __ldg(p.uniq_len + v - 1) != 1 || __ldg(p.uniq_blob + __ldg(p.uniq_off + v - 1)) != c ||
                __ldg(p.uniq_flags + v - 1) != f)
                break;
        }
    };
    if (p.one) {
        one_byte(vt[p.one + (x0 & 0xffu)]);
        if (p.nocase) one_byte(vt[p.one + 256u + (x0 & 0xffu)]);
    }
    if (room < 2) return;
    uint32_t a0 = 0, an = 0, b0 = 0, bn = 0;
    if (p.slots_a) {
        const uint32_t s = p.slots_a + 2u * (((x0 & 0xffffu) * 0x9e3779b1u) >> p.shift_a);
        a0 = vt[s]; an = vt[s + 1];
    }
    if (p.slots_b && room >= 3) {
        const uint32_t s = p.slots_b + 2u * (((x0 & 0xffffffu) * 0x9e3779b1u) >> p.shift_b);
        b0 = vt[s]; bn = vt[s + 1];
    }
    for (uint32_t r = 0; r < an + bn; r++) {
        const uint32_t *rec = vt + p.rec + 8u * (r < an ? a0 + r : b0 + (r - an));
        if ((((x0 ^ rec[0]) & rec[1]) | ((x1 ^ rec[2]) & rec[3])) != 0) continue;
        const uint32_t m = rec[4], u = rec[5];
        if (m > room || !in_window(u)) continue;
        bool same = true;
        for (uint32_t jj = 8; jj < m && same; jj += 4) { // pattern bytes jj..jj+3 against the buffer
            const uint32_t rem = m - jj;
            uint32_t diff = buf_word(buf, j + jj) ^ vt[p.blob + rec[6] + (jj >> 2)];
            if (p.nocase && rec[7]) diff &= vt[rec[7] + (jj >> 2)];
            same = (rem >= 4 ? diff : diff & ((1u << (8 * rem)) - 1u)) == 0;
        }
        if (same) window_hit<OUT>(p, s_counts, u, pos);
    }
}

template <int OUT>
__device__ __forceinline__ void window_body(const window_params &p)
{
    extern __shared__ __align__(16) uint8_t wsmem[];
    uint32_t *s_first = reinterpret_cast<uint32_t *>(wsmem);                       // [8]
    uint32_t *s_bufs = s_first + 8;                                                 // [WN_WARPS][WN_BUF_WORDS]
    uint8_t *rest = reinterpret_cast<uint8_t *>(s_bufs + WN_WARPS * WN_BUF_WORDS);
    unsigned long long *s_counts = p.counts_in_smem ? reinterpret_cast<unsigned long long *>(rest) : nullptr;
    uint32_t *s_vtab = reinterpret_cast<uint32_t *>(rest + (p.counts_in_smem ? 8u * p.n_win : 0u));
    if (threadIdx.x < 8) s_first[threadIdx.x] = p.first[threadIdx.x];
    if (s_counts)
        for (uint32_t i = threadIdx.x; i < p.n_win; i += WN_THREADS) s_counts[i] = 0;
    if (p.vtab_in_smem)
        for (uint32_t i = threadIdx.x; i < p.vtab_words; i += WN_THREADS) s_vtab[i] = __ldg(p.vtab + i);
    __syncthreads();
    const uint32_t *vt = p.vtab_in_smem ? s_vtab : p.vtab;

    const uint32_t lane = threadIdx.x & 31;
    uint32_t *buf = s_bufs + (threadIdx.x >> 5) * WN_BUF_WORDS;
    const uint64_t n_warps = (uint64_t)gridDim.x * WN_WARPS;
    for (uint64_t k = (uint64_t)blockIdx.x * WN_WARPS + (threadIdx.x >> 5); k < p.n_packets; k += n_warps) {
        const uint64_t beg = p.offsets[k], plen = p.offsets[k + 1] - beg;
        if (plen >= KMPB_PACKET_LIMIT) { // outside the documented limits (kmpb_check_device_errors reports it)
            if (lane == 0) atomicOr(p.work + 1, 1u);
            continue;
        }
        const uint32_t len = (uint32_t)plen, head = min(len, p.reach);
        const uint8_t *text = p.bytes + (beg - p.abs_base);
        uint32_t s_hi = min(p.hi_max, len == 0 ? 0u : len - 1u); // starts past it cannot fit their window or the packet
        if (len == 0 || p.lo_min > s_hi) continue;
        for (uint32_t t0 = 0; t0 <= s_hi; t0 += WN_TILE) {
            // the tile's bytes and its lookahead, [t0, t0 + need), from the 16-byte boundary below: buffer byte j is
            // packet offset t0 - lead + j
            const uint32_t need = min(head - t0, WN_TILE + WN_LOOK);
            const uint32_t lead = (uint32_t)(reinterpret_cast<uintptr_t>(text + t0) & 15u);
            const uint4 *src = reinterpret_cast<const uint4 *>(text + t0 - lead);
            const uint32_t nvec = (lead + need + 15u) / 16u;
            uint32_t z = 0xffffffffu; // first NUL, as a buffer byte
            __syncwarp();
            for (uint32_t v = lane; v < nvec; v += 32) {
                const uint4 w = __ldg(src + v);
                reinterpret_cast<uint4 *>(buf)[v] = w;
                const uint32_t ww[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
                for (uint32_t q = 0; q < 4; q++) {
                    uint32_t x = ww[q];
                    const uint32_t at = 16u * v + 4u * q;
                    if (at < lead) x |= lead - at >= 4 ? ~0u : (1u << (8u * (lead - at))) - 1u; // bytes before t0
                    const uint32_t nz = ~(((x & 0x7f7f7f7fu) + 0x7f7f7f7fu) | x) & 0x80808080u;
                    if (nz) z = min(z, at + ((uint32_t)__ffs(nz) - 1u) / 8u);
                }
            }
            z = __reduce_min_sync(0xffffffffu, z);
            __syncwarp();
            // the text ends at the packet's end or its first NUL; a NUL in this tile's range is the packet's first
            const uint32_t end = z == 0xffffffffu || z - lead >= need ? len : t0 + (z - lead);
            if (end == 0) break;
            s_hi = min(s_hi, end - 1u);
            const uint32_t o_lo = max(t0, p.lo_min), o_hi = min(s_hi, t0 + WN_TILE - 1u);
            if (o_lo <= o_hi) {
                const uint32_t w_lo = (lead + (o_lo - t0)) >> 2, w_hi = (lead + (o_hi - t0)) >> 2;
                for (uint32_t wi = w_lo + lane; wi <= w_hi; wi += 32) {
                    const uint32_t b0 = buf[wi], b1 = buf[wi + 1], b2 = buf[wi + 2];
#pragma unroll
                    for (uint32_t q = 0; q < 4; q++) {
                        const uint32_t j = 4u * wi + q, o = t0 + j - lead; // (j < lead: o wraps and fails the test)
                        if (j < lead || o < o_lo || o > o_hi) continue;
                        const uint32_t x0 = __funnelshift_r(b0, b1, 8u * q);
                        if (!(s_first[(x0 & 0xffu) >> 5] >> (x0 & 31u) & 1u)) continue;
                        const uint32_t x1 = __funnelshift_r(b1, b2, 8u * q);
                        window_probe<OUT>(p, vt, s_counts, buf, j, x0, x1, o, end - o, beg + o);
                    }
                }
            }
        } // (a NUL in the lookahead leaves the next tile the starts before it: s_hi ends the walk)
    }
    __syncthreads();
    if (s_counts)
        for (uint32_t i = threadIdx.x; i < p.n_win; i += WN_THREADS)
            if (s_counts[i]) atomicAdd(p.uniq_counts + p.u0 + i, s_counts[i]);
    if (p.n_out) { // as the union kernel's last block (union_kernel.cu), for a set without an unwindowed pattern
        __shared__ uint32_t last;
        __threadfence();
        __syncthreads();
        if (threadIdx.x == 0) {
            last = atomicAdd(p.work + 3, 1u) == gridDim.x - 1 ? 1u : 0u;
            if (last) p.work[3] = 0; // every block has counted itself in: the word is free for the next launch
        }
        __syncthreads();
        if (last) {
            __threadfence();
            for (uint32_t i = threadIdx.x; i < p.n_pat; i += WN_THREADS) {
                const unsigned long long v = __ldcg(p.uniq_counts + p.pat_to_uniq[i]);
                if (v)
                    for (uint32_t r = 0; r < p.n_out; r++) atomicAdd_system(p.out[r] + i, v);
            }
        }
    }
}

__global__ void __launch_bounds__(WN_THREADS, WN_BLOCKS_PER_SM) kmpb_window_kernel(const __grid_constant__ window_params p)
{
    window_body<WN_COUNT>(p);
}
__global__ void __launch_bounds__(WN_THREADS, WN_BLOCKS_PER_SM) kmpb_window_find_kernel(const __grid_constant__ window_params p)
{
    window_body<WN_FIND>(p);
}
__global__ void __launch_bounds__(WN_THREADS, WN_BLOCKS_PER_SM) kmpb_window_mark_kernel(const __grid_constant__ window_params p)
{
    window_body<WN_MARK>(p);
}

int kmpb_launch_window(kmpb_ctx *ctx, const kmpb_batch &b, uint32_t *d_work, uint64_t *d_uniq_counts, cudaStream_t stream,
                       const kmpb_fused_out &out, const kmpb_find_out *find, uint32_t *mark_biased)
{
    const kmpb_tables &h = ctx->host;
    const uint32_t n_win = h.n_uniq - h.n_union;
    if ((uintptr_t)b.d_bytes & 15) return kmpb_fail(KMPB_EINVAL, "payload buffer must be 16-byte aligned");
    window_params p = {};
    p.bytes = b.d_bytes;
    p.abs_base = b.abs_base;
    p.offsets = b.d_offsets;
    p.n_packets = b.n_packets;
    p.vtab = ctx->dev.wvtab;
    p.vtab_words = h.wvtab_words;
    p.slots_a = h.wvtab[1]; p.shift_a = h.wvtab[2]; p.slots_b = h.wvtab[3]; p.shift_b = h.wvtab[4];
    p.one = h.wvtab[5]; p.rec = h.wvtab[6]; p.blob = h.wvtab[7];
    p.nocase = h.win_nocase ? 1u : 0u;
    p.lo = ctx->dev.uniq_lo;
    p.hi = ctx->dev.uniq_hi;
    p.uniq_blob = ctx->dev.uniq_blob;
    p.uniq_flags = ctx->dev.uniq_flags;
    p.uniq_off = ctx->dev.uniq_off;
    p.uniq_len = ctx->dev.uniq_len;
    p.u0 = h.n_union;
    p.n_win = n_win;
    p.lo_min = h.win_lo_min;
    p.hi_max = h.win_hi_max;
    p.reach = h.win_reach;
    for (int i = 0; i < 8; i++) p.first[i] = h.win_first[i];
    p.uniq_counts = (unsigned long long *)d_uniq_counts;
    p.work = d_work;
    if (find) { p.rec_out = find->rec; p.capacity = find->capacity; p.found = find->found; }
    p.mark = mark_biased;
    p.pat_to_uniq = ctx->dev.pat_to_uniq;
    p.n_pat = h.n_pat;
    p.n_out = out.n;
    for (int r = 0; r < KMPB_MAX_OUT; r++) p.out[r] = out.vec[r];
    // the counters (64-bit) and the probe tables go into shared memory when they leave room for several blocks an SM
    const size_t fixed = 4u * (8u + WN_WARPS * WN_BUF_WORDS);
    p.counts_in_smem = 8ull * n_win <= 32768 ? 1u : 0u;
    const size_t counts_bytes = p.counts_in_smem ? 8ull * n_win : 0;
    p.vtab_in_smem = 4ull * h.wvtab_words <= 65536 ? 1u : 0u;
    const size_t smem = fixed + counts_bytes + (p.vtab_in_smem ? 4ull * h.wvtab_words : 0);
    void (*kernel)(window_params) = find ? kmpb_window_find_kernel : mark_biased ? kmpb_window_mark_kernel : kmpb_window_kernel;
    if (smem > 48 * 1024) KMPB_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const uint64_t blocks = (b.n_packets + WN_WARPS - 1) / WN_WARPS;
    const int grid = (int)std::min<uint64_t>(blocks, (uint64_t)ctx->sm_count * WN_BLOCKS_PER_SM);
    kernel<<<grid, WN_THREADS, smem, stream>>>(p);
    ctx->launches++;
    KMPB_CUDA(cudaGetLastError());
    return KMPB_OK;
}
