// perpat_kernel.cu -- the per-pattern engine (KMPB_ENGINE_PERPAT).
//
// This is the reference's packet x pattern double loop (serial.c:153-155) laid out the way
// BASELINE.json's north_star prescribes: every distinct pattern has a byte-indexed KMP transition
// DFA (built on the device, tables.cu) staged in shared memory; one warp takes one packet, cuts its
// text into 32 chunks, and every lane walks its chunk for every pattern (four patterns per walk), starting
// (pattern_len-1) bytes early so a match that straddles a chunk edge is seen by exactly one lane -- the one whose
// chunk holds the match's LAST byte.  Per-pattern hits are summed across the warp with __reduce_add_sync,
// accumulated in shared memory, and leave the block as one atomic per pattern.
//
// The packet is read from HBM once, by coalesced 16-byte loads (the scan for its first NUL), and re-walked from L1
// for every group of four patterns, so this engine is bound by instruction issue (~P x 5.5 instructions per byte),
// not by HBM; it exists as the literal form of the design, as an independent on-device cross-check of the union
// engine, and for the DFA-shared-memory-pressure sweep (BASELINE config 4).  Pattern sets whose DFAs exceed shared
// memory are processed in tiles, one launch per tile.
#include <algorithm>

#include "kmpb_device.cuh"

constexpr int PP_THREADS = 1024;

constexpr int PP_GROUP = 4; // patterns per walk

// One lane's walk over its chunk [a, stop) of a text for NP (1..PP_GROUP) patterns at once -> hits[] whose last byte
// lies in the chunk.  One DFA step: entry = rows[256 * state + byte] = next state | hit << 7; `sp` is the shared
// address of the current state's row, so a step is: add the byte, load, count bit 7, rebuild the row address.  The
// automata step on the same text bytes, and NP independent chains of (shared-memory load -> next row address) per
// lane hide each other's latency.  mm = the longest pattern's length.
template <int NP>
__device__ __forceinline__ void walk_chunk(const uint8_t *text, const uint32_t a, const uint32_t stop, const uint32_t mm,
                                          const uint32_t (&rows)[PP_GROUP], uint32_t (&hits)[PP_GROUP])
{
    uint32_t sp[NP];
#pragma unroll
    for (int k = 0; k < NP; k++) sp[k] = rows[k];
    auto step = [&](uint32_t byte) {
        uint32_t e[NP];
#pragma unroll
        for (int k = 0; k < NP; k++) asm("ld.shared.u8 %0, [%1];" : "=r"(e[k]) : "r"(sp[k] + byte));
#pragma unroll
        for (int k = 0; k < NP; k++) {
            hits[k] += e[k] >> 7;
            sp[k] = rows[k] + ((e[k] & 0x7fu) << 8);
        }
    };
    // run-in: the (m - 1) bytes before the chunk only bring the automaton into its state (a KMP state depends on the
    // last m - 1 bytes at most, so starting earlier for the shorter patterns changes nothing); a hit there has its last
    // byte in the previous lane's chunk and is that lane's
    uint32_t i = a >= mm - 1 ? a - (mm - 1) : 0;
    for (; i < a; i++) step(text[i]);
#pragma unroll
    for (int k = 0; k < NP; k++) hits[k] = 0;
    // the chunk: bytes up to the next word boundary, whole words (L1-resident after the NUL scan, one load per four
    // steps), the rest
    const uintptr_t text_addr = reinterpret_cast<uintptr_t>(text);
    for (; i < stop && ((text_addr + i) & 3u); i++) step(text[i]);
    for (; i + 4 <= stop; i += 4) {
        const uint32_t w = __ldg(reinterpret_cast<const uint32_t *>(text + i));
        step(w & 0xffu);
        step(__byte_perm(w, 0, 0x4441));
        step(__byte_perm(w, 0, 0x4442));
        step(w >> 24);
    }
    for (; i < stop; i++) step(text[i]);
}

__global__ void __launch_bounds__(PP_THREADS, 1)
kmpb_perpat_kernel(const uint8_t *__restrict__ bytes, uint64_t abs_base, const uint64_t *__restrict__ offsets,
                   uint64_t n_packets, const uint8_t *__restrict__ dfa_all, const uint32_t *__restrict__ uniq_off,
                   uint32_t u0, uint32_t u1, unsigned long long *__restrict__ uniq_counts)
{
    extern __shared__ __align__(16) uint8_t smem[];
    const uint32_t n_tile = u1 - u0;
    uint32_t *s_counts = reinterpret_cast<uint32_t *>(smem);            // [n_tile]
    uint32_t *s_off = s_counts + n_tile;                                 // [n_tile+1], relative to the tile
    uint8_t *s_dfa = smem + ((8u * n_tile + 4u + 15u) & ~15u);           // tile's DFA rows, 256 B each

    const uint32_t tile_base = uniq_off[u0];
    for (uint32_t i = threadIdx.x; i <= n_tile; i += PP_THREADS) {
        s_off[i] = uniq_off[u0 + i] - tile_base;
        if (i < n_tile) s_counts[i] = 0;
    }
    {   // stage the DFA rows with 16-byte loads (rows are 256-byte multiples, 256-byte aligned)
        const uint4 *src = reinterpret_cast<const uint4 *>(dfa_all + 256ull * tile_base);
        uint4 *dst = reinterpret_cast<uint4 *>(s_dfa);
        const uint32_t n16 = (uniq_off[u1] - tile_base) * 16u;
        for (uint32_t i = threadIdx.x; i < n16; i += PP_THREADS) dst[i] = src[i];
    }
    __syncthreads();

    const uint32_t lane = threadIdx.x & 31;
    const uint64_t warp = (uint64_t)blockIdx.x * (PP_THREADS / 32) + (threadIdx.x >> 5);
    const uint64_t n_warps = (uint64_t)gridDim.x * (PP_THREADS / 32);

    for (uint64_t k = warp; k < n_packets; k += n_warps) {
        const uint64_t beg = offsets[k];
        const uint32_t len = (uint32_t)(offsets[k + 1] - beg);
        const uint8_t *text = bytes + (beg - abs_base);
        // The text ends at the first NUL byte (strlen in kmp_matcher, serial.c:191).  Coalesced 16-byte loads from
        // the 16-byte boundary below the packet's start, four per lane in flight (2 KB per warp trip), so that a
        // 1400-byte packet is one round trip to memory instead of one per 32 bytes; the warp stops at the first
        // trip that holds a NUL.  The batch is readable up to the next multiple of 16 (include/kmpb200.h).
        const uint32_t lead = (uint32_t)((beg - abs_base) & 15u);
        const uint4 *vec = reinterpret_cast<const uint4 *>(text - lead);
        const uint32_t nvec = (lead + len + 15u) / 16u;
        uint32_t z = len;
        for (uint32_t v0 = 0; v0 < nvec; v0 += 128) {
            uint4 w[4];
#pragma unroll
            for (uint32_t j = 0; j < 4; j++) {
                const uint32_t v = v0 + 32 * j + lane;
                w[j] = v < nvec ? __ldg(vec + v) : make_uint4(~0u, ~0u, ~0u, ~0u);
            }
#pragma unroll
            for (uint32_t j = 0; j < 4; j++) {
                const uint32_t v = v0 + 32 * j + lane;
                const uint32_t ww[4] = {w[j].x, w[j].y, w[j].z, w[j].w};
#pragma unroll
                for (uint32_t q = 0; q < 4; q++) {
                    uint32_t x = ww[q];
                    const uint32_t at = 16u * v + 4u * q; // position of this word's first byte, from text - lead
                    if (at < lead) x |= lead - at >= 4 ? ~0u : (1u << (8u * (lead - at))) - 1u; // bytes before the packet
                    // bit 7 of every byte that is zero (exact per byte: no carries between bytes)
                    const uint32_t nz = ~(((x & 0x7f7f7f7fu) + 0x7f7f7f7fu) | x) & 0x80808080u;
                    if (nz) z = min(z, at + ((uint32_t)__ffs(nz) - 1u) / 8u - lead); // at + byte >= lead here
                }
            }
            if (__any_sync(0xffffffffu, z < len)) break;
        }
        const uint32_t n = min(len, __reduce_min_sync(0xffffffffu, z));
        if (n == 0) continue;
        const uint32_t chunk = (n + 31) / 32;
        const uint32_t a = lane * chunk;
        const uint32_t stop = min(a + chunk, n);
        // PP_GROUP patterns per walk (walk_chunk)
        for (uint32_t t = 0; t < n_tile; t += PP_GROUP) {
            const uint32_t np = n_tile - t < (uint32_t)PP_GROUP ? n_tile - t : (uint32_t)PP_GROUP;
            uint32_t hits[PP_GROUP] = {0, 0, 0, 0};
            if (a < n) { // (a pattern longer than the text cannot hit: "no point trying to match things", serial.c:193)
                uint32_t rows[PP_GROUP], mm = 0;
#pragma unroll
                for (uint32_t k = 0; k < (uint32_t)PP_GROUP; k++) {
                    const uint32_t u = t + (k < np ? k : 0);
                    rows[k] = (uint32_t)__cvta_generic_to_shared(s_dfa + 256u * s_off[u]);
                    mm = max(mm, s_off[u + 1] - s_off[u]);
                }
                if (np == 4) walk_chunk<4>(text, a, stop, mm, rows, hits);
                else if (np == 3) walk_chunk<3>(text, a, stop, mm, rows, hits);
                else if (np == 2) walk_chunk<2>(text, a, stop, mm, rows, hits);
                else walk_chunk<1>(text, a, stop, mm, rows, hits);
            }
#pragma unroll
            for (uint32_t k = 0; k < (uint32_t)PP_GROUP; k++) {
                if (k < np) { // warp-uniform
                    const uint32_t total = __reduce_add_sync(0xffffffffu, hits[k]);
                    if (lane == 0 && total) atomicAdd(&s_counts[t + k], total);
                }
            }
        }
    }
    __syncthreads();
    for (uint32_t t = threadIdx.x; t < n_tile; t += PP_THREADS)
        if (s_counts[t]) atomicAdd(&uniq_counts[u0 + t], (unsigned long long)s_counts[t]);
}

// The windowed patterns (distinct ids [u0, u0 + n_win), kmpb_set_patterns_win): each by its own DFA walk over the bytes
// [lo, hi + m) of every packet's text, from the start state at lo, so that a hit is a match that starts in [lo, hi].  One
// warp per packet: the text's end (its first NUL) among the first `reach` bytes, then per pattern the 32 lanes walk a
// chunk each of that range, with the run-in of walk_chunk clipped at lo.  It shares nothing with the window kernel
// (window.cu) or its tables, so it stays an independent cross-check of it.
constexpr int PPW_THREADS = 256;
__global__ void __launch_bounds__(PPW_THREADS)
kmpb_perpat_window_kernel(const uint8_t *__restrict__ bytes, uint64_t abs_base, const uint64_t *__restrict__ offsets,
                          uint64_t n_packets, const uint8_t *__restrict__ dfa_all, const uint32_t *__restrict__ uniq_off,
                          const uint32_t *__restrict__ win_lo, const uint32_t *__restrict__ win_hi, uint32_t u0, uint32_t n_win,
                          uint32_t reach, unsigned long long *__restrict__ uniq_counts)
{
    const uint32_t lane = threadIdx.x & 31;
    const uint64_t n_warps = (uint64_t)gridDim.x * (PPW_THREADS / 32);
    for (uint64_t k = (uint64_t)blockIdx.x * (PPW_THREADS / 32) + (threadIdx.x >> 5); k < n_packets; k += n_warps) {
        const uint64_t beg = offsets[k];
        const uint32_t head = (uint32_t)min(offsets[k + 1] - beg, (uint64_t)reach);
        const uint8_t *text = bytes + (beg - abs_base);
        uint32_t z = head;
        for (uint32_t i = lane; i < head; i += 32)
            if (text[i] == 0) { z = i; break; }
        const uint32_t n = __reduce_min_sync(0xffffffffu, z);
        for (uint32_t w = 0; w < n_win; w++) {
            const uint32_t u = u0 + w, m = uniq_off[u + 1] - uniq_off[u], lo = win_lo[w];
            const uint32_t e = min(win_hi[w] + m, n);
            if (lo + m > e) continue; // (warp-uniform)
            const uint32_t chunk = (e - lo + 31) / 32, a = lo + lane * chunk, stop = min(a + chunk, e);
            const uint8_t *rows = dfa_all + 256ull * uniq_off[u];
            uint32_t hits = 0;
            if (a < e) {
                uint32_t state = 0;
                for (uint32_t i = a >= lo + (m - 1) ? a - (m - 1) : lo; i < stop; i++) {
                    const uint32_t entry = __ldg(rows + 256u * state + text[i]);
                    if (i >= a) hits += entry >> 7;
                    state = entry & 0x7fu;
                }
            }
            const uint32_t total = __reduce_add_sync(0xffffffffu, hits);
            if (lane == 0 && total) atomicAdd(&uniq_counts[u], (unsigned long long)total);
        }
    }
}

int kmpb_launch_perpat(kmpb_ctx *ctx, const kmpb_batch &b, uint64_t *d_uniq_counts, cudaStream_t stream)
{
    const kmpb_tables &h = ctx->host;
    if (h.n_uniq == 0 || b.n_packets == 0) return KMPB_OK;
    if ((uintptr_t)b.d_bytes & 15) return kmpb_fail(KMPB_EINVAL, "payload buffer must be 16-byte aligned"); // 16-byte loads
    const size_t budget = ctx->smem_optin;
    if (!ctx->attr_perpat_set) {
        KMPB_CUDA(cudaFuncSetAttribute(kmpb_perpat_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)budget));
        ctx->attr_perpat_set = true;
    }
    if (h.n_union < h.n_uniq) { // the windowed patterns
        if (ctx->profile) KMPB_CUDA(cudaEventRecord(ctx->ev_kernel[0], stream));
        const int grid = (int)std::min<uint64_t>((uint64_t)ctx->sm_count * 8, (b.n_packets + PPW_THREADS / 32 - 1) / (PPW_THREADS / 32));
        kmpb_perpat_window_kernel<<<grid, PPW_THREADS, 0, stream>>>(
            b.d_bytes, b.abs_base, b.d_offsets, b.n_packets, ctx->dev.perpat_dfa, ctx->dev.uniq_off, ctx->dev.uniq_lo,
            ctx->dev.uniq_hi, h.n_union, h.n_uniq - h.n_union, h.win_reach, (unsigned long long *)d_uniq_counts);
        ctx->launches++;
        KMPB_CUDA(cudaGetLastError());
    }
    uint32_t u0 = 0;
    while (u0 < h.n_union) {
        // largest tile [u0, u1) whose counters + offsets + DFA rows fit
        uint32_t u1 = u0;
        size_t need = 0;
        while (u1 < h.n_union) {
            uint32_t nt = u1 + 1 - u0;
            size_t want = ((8u * nt + 4u + 15u) & ~15u) + 256ull * (h.uniq_off[u1 + 1] - h.uniq_off[u0]);
            if (want > budget) break;
            need = want;
            u1++;
        }
        if (u1 == u0) return kmpb_fail(KMPB_ELIMIT, "pattern %u does not fit in shared memory", u0);
        uint64_t warps_wanted = b.n_packets;
        int grid = (int)std::min<uint64_t>((uint64_t)ctx->sm_count, (warps_wanted + PP_THREADS / 32 - 1) / (PP_THREADS / 32));
        if (ctx->profile && u0 == 0 && h.n_union == h.n_uniq) KMPB_CUDA(cudaEventRecord(ctx->ev_kernel[0], stream));
        kmpb_perpat_kernel<<<grid, PP_THREADS, need, stream>>>(b.d_bytes, b.abs_base, b.d_offsets, b.n_packets,
                                                               ctx->dev.perpat_dfa, ctx->dev.uniq_off, u0, u1,
                                                               (unsigned long long *)d_uniq_counts);
        ctx->launches++;
        KMPB_CUDA(cudaGetLastError());
        u0 = u1;
    }
    if (ctx->profile) KMPB_CUDA(cudaEventRecord(ctx->ev_kernel[1], stream));
    return KMPB_OK;
}
