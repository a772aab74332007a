// union_kernel.cu -- the union engine (KMPB_ENGINE_UNION): every payload byte is read from HBM once.
//
// Two levels, strictly separated.
//
//  FAST PATH (every byte) knows nothing about packets.  A warp streams work items -- runs of whole
//  packets, ~64 KB of the flat CSR byte buffer -- in rows of 1024 contiguous bytes.  A row travels
//  global -> registers by ONE coalesced 256-bit load per lane (SASS LDG.E.256, L1 not allocated): lane l
//  holds bytes [32 l, 32 l + 32) of the row in eight registers; UN_NBUF such row buffers rotate (the loop is
//  unrolled UN_NBUF times, so the rotation costs no moves) and an L2 prefetch runs UN_PF rows ahead of the
//  loads.  The four bytes a lane needs after its own come from the next lane's first register (one SHFL); lane
//  31 loads the four bytes after the row itself.  (Round 1 staged the rows in a shared-memory ring filled by
//  cp.async: ring write + read-back cost 17-28 shared-memory wavefronts per row next to the filter's 35.)
//  Each lane pushes its 32 bytes (+4 bytes of lookahead) through a 4-byte-deep shift-and filter over 5 pattern
//  buckets and a NUL detector, in 6-bit fields with a fifth field in which a report lingers one step, so that
//  the state is updated once per TWO bytes:
//      S = ((S << 12) | 0xfff) & G[b0] & L[b1],      G[c] = (L[c] << 6) | 0x3f
//  L and G live in shared memory in a bank-private layout (byte address = byte * 128 + lane * 4), so the one
//  lookup per byte never bank-conflicts; its address is one IDP.4A (byte x 128 + lane base: the FMA pipe, which
//  this integer kernel otherwise leaves idle; round 1 built the address with a PRMT on the ALU pipe, the busiest
//  one, and needed a 64 KB-aligned table for it).  The shift-or is one integer multiply-add (FMA pipe), the
//  three-way AND one LOP3 (ALU pipe).  After an update bits 24..28 say "the 4 bytes ending at b0 are the first 4
//  bytes (or all the bytes) of some pattern of bucket b", bits 18..22 the same for b1; bits 29 / 23 say "the
//  byte three before b0 / b1 is NUL" (the NUL detector reports as late as a pattern that starts at the NUL
//  would, which keeps "what starts here" and "is this a NUL" of a byte in the same report).  The reports are
//  OR-ed per quarter of the group (8 start positions); a lane with any report appends an EVENT -- eight bytes: which
//  group of the item it is (| the item's parity << 31) and which quarters reported what -- to the warp's ring in
//  shared memory.  That is all: one ballot and one 8-byte store per reporting lane on top of the filter.  An event
//  carries no text: the resolve step fetches the 36 bytes it needs again, from L2 (the row was read a few
//  microseconds ago), which is cheaper than writing 48 bytes per event from the row loop and keeps the loop's
//  registers free of the lookahead words.  (NUL-dense rows: events that hold only NULs and are superseded by a
//  later one of the same row are dropped first, drop_superseded.)
//
//  SLOW PATH (events only).  The ring has UN_QCAP slots; whenever it holds 32 events, the warp -- at the top of the
//  row loop, the ONE place the resolve step is inlined (a call from inside the loop made ptxas spill five of the
//  loop's values around it; the item switch and the final flush call a not-inlined copy) -- resolves the 32 oldest
//  at once, in stream order, one per lane:
//  Phase 0 (issued one trip of the row loop earlier, cp.async: nobody waits for L2): the lane's event's group (32 B,
//  and 8 B of lookahead when its last quarter reported) travels into the warp's staging area.  (One bulk copy -- TMA --
//  per event completing on a per-warp mbarrier was measured in its place: 13 % slower, 48-byte copies are not what that
//  engine is for.)
//  Phase 1:
//    - the lane re-runs the filter over the quarter that reported (two bytes per update, like the row loop), this time
//      recording which start positions fired and which bytes are NUL;
//    - it finds the packet that holds its first candidate: a division when all the item's packets have the same size,
//      else a search in the item's slice of `offsets` (interpolation guess, then binary search); the item's packet and
//      byte range waits in the warp's scratch words;
//    - a candidate start q in packet [ps, pe) is alive when no NUL lies in [ps, q) -- the reference's
//      "text ends at the first NUL" rule (serial.c:191).  NULs inside the quarter come from the lane's own
//      mask; the last NUL before it comes from the nearest earlier event that held one (events are in
//      stream order, every NUL byte of the stream raises one) or from the warp's carry.
//  Phase 2: every lane appends its alive candidates -- first 8 text bytes, absolute position, bytes left in the packet:
//  16 bytes, self-contained -- to the warp's CANDIDATE RING, at its own pace (slot runs from a prefix sum of the counts).
//  Whenever 32 candidates are waiting, whichever resolve step they came from, they are verified one per lane: the
//  candidate's first bytes select one slot in each of the two probe tables of automaton.c (two-byte patterns by their
//  two bytes, longer ones by their first three), the slots' pattern records (first 8 bytes + masks, length, id) are
//  compared, longer patterns word by word against the text in global memory, and a hit is counted when it ends inside
//  its packet (q + len <= pe).  Every verification round runs with all 32 lanes busy; what is left at the end of the
//  batch is flushed.
//  So every pattern occurrence that lies inside one packet and has no NUL before it in that packet is
//  counted exactly once.  Counts go to shared-memory counters and leave the block as one atomic per
//  distinct pattern.  No separators, no padding and no second pass over the payload.
#include <algorithm>
#include <cooperative_groups.h>
#include <type_traits>

#include "kmpb_device.cuh"

#ifndef KMPB_UN_THREADS
#define KMPB_UN_THREADS 1024
#endif
#ifndef KMPB_UN_ITEM_KB
#define KMPB_UN_ITEM_KB 64
#endif
#ifndef KMPB_UN_NBUF
#define KMPB_UN_NBUF 2
#endif
#ifndef KMPB_UN_PF
#define KMPB_UN_PF 6
#endif
constexpr int UN_THREADS = KMPB_UN_THREADS; // one block per SM
constexpr int UN_WARPS = UN_THREADS / 32;
constexpr uint32_t UN_GRP = 32;                           // bytes per lane per row
constexpr uint32_t UN_ROW = 32 * UN_GRP;                  // bytes per warp row
constexpr uint32_t UN_NBUF = KMPB_UN_NBUF;                // row buffers (registers) per lane: UN_NBUF - 1 rows in flight
constexpr uint32_t UN_PF = KMPB_UN_PF;                    // rows the L2 prefetch runs ahead of the loads (0: none)
static_assert(UN_NBUF >= 2 && UN_NBUF <= 4, "2..4 row buffers");
constexpr uint32_t UN_ITEM_BYTES = KMPB_UN_ITEM_KB << 10; // target work-item size
#ifndef KMPB_UN_TAIL_ITEMS
#define KMPB_UN_TAIL_ITEMS 16384
#endif
constexpr uint32_t UN_TAIL_ITEMS = KMPB_UN_TAIL_ITEMS;   // small items at the end of a batch (about one per warp x 4)
constexpr uint32_t UN_QCAP = 128;   // slots of a warp's event ring (fewer than 32 pending + at most 32 of each of two rows)
#ifndef KMPB_UN_QDRAIN
#define KMPB_UN_QDRAIN 32
#endif
constexpr uint32_t UN_QDRAIN = KMPB_UN_QDRAIN; // events resolved at once (one per lane)
static_assert(UN_QDRAIN >= 8 && UN_QDRAIN <= 32, "one event per lane");
constexpr uint32_t UN_Q_BYTES1 = 8; // an event in the ring: group index | item parity << 31, quarter reports
constexpr uint32_t UN_T_WORDS = 12; // an event being resolved: 32 B group, 8 B lookahead, group index | parity, packet boundaries in the group
constexpr uint32_t UN_T_BYTES1 = UN_T_WORDS * 4;
#ifndef KMPB_UN_DENSE
#define KMPB_UN_DENSE 12
#endif
constexpr uint32_t UN_DENSE = KMPB_UN_DENSE; // reporting groups per row from which superseded NUL-only events are dropped (> 32: never)
constexpr uint32_t UN_LUT_BYTES = 256 * 128; // one table: a 128-byte row (32 lanes x 4 bytes) per byte value
constexpr uint32_t FULL = 0xffffffffu;

// Dynamic shared memory: L, G, the event rings, the events being resolved, the warps' scratch words, the counters (if
// they fit), the probe tables (if they fit).
constexpr uint32_t UN_Q_BYTES = UN_WARPS * UN_QCAP * UN_Q_BYTES1;
constexpr uint32_t UN_T_BYTES = UN_WARPS * UN_QDRAIN * UN_T_BYTES1; // the 32 events a warp is resolving, with their text
constexpr uint32_t UN_CCAP = 128;     // slots of a warp's candidate ring: fewer than 32 waiting + what a resolve step finds (else: trips of 32)
constexpr uint32_t UN_C_BYTES1 = 16;  // a candidate: its first 8 text bytes, its absolute position, the bytes left in its packet
constexpr uint32_t UN_C_BYTES = UN_WARPS * UN_CCAP * UN_C_BYTES1;
constexpr uint32_t UN_SCRATCH_BYTES = UN_WARPS * 128;
constexpr uint32_t UN_OFF_Q = 2 * UN_LUT_BYTES;
constexpr uint32_t UN_OFF_T = UN_OFF_Q + UN_Q_BYTES;
constexpr uint32_t UN_OFF_C = UN_OFF_T + UN_T_BYTES;       // the warps' candidate rings
constexpr uint32_t UN_OFF_SCRATCH = UN_OFF_C + UN_C_BYTES;
constexpr uint32_t UN_OFF_MISC = UN_OFF_SCRATCH + UN_SCRATCH_BYTES; // 128 bytes: what the resolve step reads of the
                                                                    // launch parameters (DC_*), the "last block" flag
constexpr uint32_t UN_OFF_COUNTS = UN_OFF_MISC + 128;
constexpr size_t UN_SMEM_FIXED = UN_OFF_COUNTS;
constexpr size_t UN_SMEM_MAX = 227 * 1024; // opt-in shared memory of one block on sm_100
static_assert(UN_SMEM_FIXED + 12288 <= UN_SMEM_MAX, "shared memory budget");

// the filter's geometry (automaton.c kmpb_filter6_build): fields of 6 bits, bits 0..4 the pattern buckets, bit 5 the NUL
// detector; after a two-byte update b0's reports sit in bits 24..29, b1's in bits 18..23
constexpr uint32_t F6_HI = 0x3f000000u, F6_LO = 0x00fc0000u;

struct union_params {
    const uint8_t *bytes; // device pointer to absolute byte abs_base (abs_base % 512 == 0)
    uint64_t abs_base;
    const uint64_t *offsets; // [n_packets+1], absolute
    uint32_t n_packets;
    const uint32_t *items; // [n_items+1] first packet of each work item
    uint32_t n_items;
    uint32_t *work;         // [0] next item, [1] error flags (until kmpb_check_device_errors), [2] blocks that have finished
    const uint32_t *filter; // [256] filter words in 6-bit fields
    uint32_t n_uniq;
    uint32_t counts_in_smem; // counters live in shared memory
    uint32_t vtab_in_smem;   // the probe tables live in shared memory
    const uint32_t *vtab;    // probe tables (automaton.c build_verify_tables); the header words follow as scalars
    uint32_t vtab_words;
    uint32_t vt_slots_a, vt_shift_a, vt_slots_b, vt_shift_b, vt_one, vt_rec, vt_blob;
    uint32_t mul64, mul4096; // the values 64 and 4096, passed at run time so that the shift-ors compile to integer
                             // multiply-adds on the FMA pipe instead of competing for the ALU pipe
    uint32_t sel[4];         // 0x80 << 8k: the IDP.4A's byte selectors, read from the constant bank by the instruction
                             // itself (as immediates they cost the row loop four UMOVs per row)
    unsigned long long *uniq_counts;
    // fused expansion + reduction (n_out > 0): the last block to finish adds every pattern's count, in file
    // order, to out[0..n_out) -- this GPU's count vector and/or its peers' (NVLink-mapped)
    const uint32_t *pat_to_uniq;
    uint32_t n_pat, n_out;
    unsigned long long *out[KMPB_MAX_OUT];
};

// ---- work partition: item i = packets [items[i], items[i+1]) ---------------------------------
// It also flags (work[1]) every packet of KMPB_PACKET_LIMIT bytes or more: such a packet runs across some item's target,
// as targets lie at most an item apart, and it is the packet just before that item's first.
__global__ void kmpb_union_partition_kernel(const uint64_t *__restrict__ offsets, uint32_t n_packets,
                                            uint32_t n_items, uint32_t n_big, uint64_t item_bytes, uint64_t small_bytes,
                                            uint32_t *__restrict__ items,
                                            uint32_t *__restrict__ work)
{
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0) { work[0] = 0; work[2] = 0; }
    if (i > n_items) return;
    if (i == n_items) { items[i] = n_packets; return; }
    // first packet whose start is >= the item's target byte: n_big items of item_bytes, then small
    // items, so that the warps run dry within a small item of each other at the end of the batch
    const uint64_t target = offsets[0] + (i <= n_big ? (uint64_t)i * item_bytes
                                                     : (uint64_t)n_big * item_bytes + (uint64_t)(i - n_big) * small_bytes);
    // guess by the mean packet size (exact for equal-sized packets), bracket the answer by doubling steps around the
    // guess, then bisect: a few dependent loads instead of log2(n_packets)
    const uint64_t first = offsets[0], total = offsets[n_packets] - first;
    uint32_t lo = 0, hi = n_packets;
    if (total) {
        const double frac = (double)(target - first) / (double)total;
        uint32_t g = (uint32_t)(frac * (double)n_packets);
        g = g > n_packets ? n_packets : g;
        if (offsets[g] < target) { // the answer lies above g
            lo = g + 1;
            for (uint32_t step = 1; lo < n_packets; step *= 2) {
                const uint32_t probe = lo + step - 1 < n_packets ? lo + step - 1 : n_packets;
                if (offsets[probe] >= target) { hi = probe; break; }
                lo = probe + 1;
                if (probe == n_packets) break;
            }
            if (lo > hi) lo = hi;
        } else { // at or below g
            hi = g;
            for (uint32_t step = 1; hi > 0; step *= 2) {
                const uint32_t probe = hi > step ? hi - step : 0;
                if (offsets[probe] < target) { lo = probe + 1; break; }
                hi = probe;
            }
        }
    }
    while (lo < hi) {
        uint32_t mid = lo + (hi - lo) / 2;
        if (offsets[mid] < target) lo = mid + 1; else hi = mid;
    }
    items[i] = lo;
    if (lo > 0 && offsets[lo] - offsets[lo - 1] >= KMPB_PACKET_LIMIT) atomicOr(work + 1, 1u);
}

// ---- helpers -----------------------------------------------------------------------------------
// One row buffer of a lane: its 32 bytes of a row.
struct row_regs {
    uint32_t w[8];
};
// 32 bytes global -> registers in one instruction (SASS LDG.E.256, sm_100), L1 not allocated (the row is used once).
// Unconditional, into pure outputs: a predicated load has to keep the registers' old values, and ptxas then loads
// into temporaries and moves (eight moves per row) once the load sits in the middle of another row's scan.
__device__ __forceinline__ void ldg256(row_regs &b, const void *src)
{
    asm volatile("ld.global.L1::no_allocate.v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(b.w[0]), "=r"(b.w[1]), "=r"(b.w[2]), "=r"(b.w[3]), "=r"(b.w[4]), "=r"(b.w[5]), "=r"(b.w[6]), "=r"(b.w[7])
                 : "l"(src));
}
// 4 bytes under a predicate (lane 31's lookahead); 0 otherwise
__device__ __forceinline__ uint32_t ldg32_if(bool on, const void *src)
{
    uint32_t v;
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %2, 0;\n\tmov.u32 %0, 0;\n\t"
                 "@p ld.global.L1::no_allocate.u32 %0, [%1];\n\t}"
                 : "=&r"(v)
                 : "l"(src), "r"((uint32_t)on));
    return v;
}
// the 128-byte line at src on its way into L2 (SASS CCTL.E.PF2): no registers, no wait
__device__ __forceinline__ void prefetch_l2_if(bool on, const void *src)
{
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %1, 0;\n\t@p prefetch.global.L2 [%0];\n\t}" ::"l"(src), "r"((uint32_t)on) : "memory");
}
template <uint32_t OFF>
__device__ __forceinline__ void prefetch_l2_if(bool on, const void *src)
{
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %1, 0;\n\t@p prefetch.global.L2 [%0+%2];\n\t}" ::"l"(src), "r"((uint32_t)on), "n"(OFF) : "memory");
}
// pointer + 32-bit offset as IMAD.WIDE.U32 (FMA pipe), not IADD3 + IADD3.X (ALU pipe)
__device__ __forceinline__ const uint8_t *add_wide(const uint8_t *base, uint32_t offset)
{
    uint64_t r;
    asm("mad.wide.u32 %0, %1, 1, %2;" : "=l"(r) : "r"(offset), "l"(reinterpret_cast<uint64_t>(base)));
    return reinterpret_cast<const uint8_t *>(r);
}
__device__ __forceinline__ uint4 lds128v(uint32_t saddr)
{
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(saddr) : "memory");
    return v;
}
// loads through 32-bit shared addresses (read-only tables, or data ordered by __syncwarp)
__device__ __forceinline__ uint32_t lds32(uint32_t saddr)
{
    uint32_t v;
    asm("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(saddr));
    return v;
}
// the same address in table G (one table further on): an immediate offset, no second base register
__device__ __forceinline__ uint32_t lds32_g(uint32_t saddr)
{
    uint32_t v;
    asm("ld.shared.u32 %0, [%1+32768];" : "=r"(v) : "r"(saddr));
    return v;
}
__device__ __forceinline__ uint2 lds64(uint32_t saddr)
{
    uint2 v;
    asm("ld.shared.v2.u32 {%0,%1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(saddr));
    return v;
}
__device__ __forceinline__ uint4 lds128(uint32_t saddr)
{
    uint4 v;
    asm("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(saddr));
    return v;
}
__device__ __forceinline__ uint2 lds64v(uint32_t saddr)
{
    uint2 v;
    asm volatile("ld.shared.v2.u32 {%0,%1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(saddr) : "memory");
    return v;
}
__device__ __forceinline__ uint32_t lds32v(uint32_t saddr)
{
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(saddr) : "memory");
    return v;
}
__device__ __forceinline__ void sts32v(uint32_t saddr, uint32_t a)
{
    asm volatile("st.shared.u32 [%0], %1;" ::"r"(saddr), "r"(a) : "memory");
}
__device__ __forceinline__ void sts64v(uint32_t saddr, uint32_t a, uint32_t b)
{
    asm volatile("st.shared.v2.u32 [%0], {%1,%2};" ::"r"(saddr), "r"(a), "r"(b) : "memory");
}
__device__ __forceinline__ void sts128v(uint32_t saddr, uint32_t a, uint32_t b, uint32_t c, uint32_t d)
{
    asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(saddr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
// global -> shared without a register in between (SASS LDGSTS); `bytes` of the 16 (8) are read, the rest is zero-filled
__device__ __forceinline__ void cp_async16(uint32_t saddr, const void *src, uint32_t bytes)
{
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(saddr), "l"(src), "r"(bytes) : "memory");
}
__device__ __forceinline__ void cp_async8(uint32_t saddr, const void *src, uint32_t bytes)
{
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;" ::"r"(saddr), "l"(src), "r"(bytes) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }
__device__ __forceinline__ void sts8v(uint32_t saddr, uint32_t a) { asm volatile("st.shared.u8 [%0], %1;" ::"r"(saddr), "r"(a) : "memory"); }
__device__ __forceinline__ uint32_t lds8v(uint32_t saddr)
{
    uint32_t v;
    asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(saddr) : "memory");
    return v;
}
__device__ __forceinline__ uint32_t saddr_of(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

// bits [0, x) of a 32-bit word, 0 <= x <= 32 (PTX shl clamps a shift amount above 31 to 32: 1 << 32 is 0, minus 1 all ones)
__device__ __forceinline__ uint32_t bits_below(uint32_t x)
{
    uint32_t r;
    asm("shl.b32 %0, 1, %1;" : "=r"(r) : "r"(x));
    return r - 1u;
}
// bits [lo, hi) of a 32-bit word, 0 <= lo, hi <= 32
__device__ __forceinline__ uint32_t bit_window(uint32_t lo, uint32_t hi) { return bits_below(hi) & ~bits_below(lo); }
// x clamped to 0..32, x signed
__device__ __forceinline__ uint32_t clamp32(int32_t x) { return (uint32_t)min(max(x, 0), 32); }

// filter words of byte k (0..3) of `word`: the IDP.4A builds the whole shared address, byte * 128 + the lane's base
// in table L (lutL) or G (lutG)
#define LUT_L(word, k) lds32(__dp4a((uint32_t)(word), DP_SEL(k), lutL))
#define LUT_G(word, k) lds32_g(__dp4a((uint32_t)(word), DP_SEL(k), lutL))
#define DP_SEL(k) (0x80u << (8 * (k))) // 128 x byte k
// one two-byte update: bytes k0, k1 = k0 + 1 of `word`
#define SA2(word, k0) (S = (S * mul2 + 4095u) & LUT_G(word, k0) & LUT_L(word, (k0) + 1))

// The launch parameters the resolve step reads, copied to shared memory once per block (word indices in the block at
// UN_OFF_MISC): a function that is not inlined would reach the kernel's parameter space through generic loads.
enum { DC_TEXT_LO = 0, DC_TEXT_HI,   // p.bytes - p.abs_base: absolute byte 0
       DC_OFF_LO, DC_OFF_HI,     // p.offsets
       DC_VTAB_LO, DC_VTAB_HI,   // p.vtab (global)
       DC_CNT_LO, DC_CNT_HI,     // p.uniq_counts
       DC_SLOTS_A, DC_SHIFT_A, DC_SLOTS_B, DC_SHIFT_B, DC_ONE, DC_REC, DC_BLOB,
       DC_MUL4096, DC_VTAB_SA,     // shared address of the probe tables, 0 = they are in global memory
       DC_COUNTS_SA,             // shared address of the counters, 0 = global atomics
       DC_REC_LO = 18, DC_REC_HI, // find kernel: the record buffer (kmpb_match[capacity])
       DC_CAP_LO, DC_CAP_HI,     // ... its capacity in records
       DC_FOUND_LO, DC_FOUND_HI, // ... the uint64 counter of every match found (also those past the capacity)
       DC_LAST = 31 };           // "I am the last block" flag

// The scratch words of a warp (128 bytes): two sets of 32 bytes, one per item parity --
//   {ks (or 1 / L as a float when all packets have L bytes), ke, b_rel, e_rel, row0 lo, row0 hi, carry, packet size}: the item's packets [ks, ke), its bytes
//   [b_rel, e_rel) relative to row0 = the absolute position of its first row, 1 + the (relative) position of the last
//   NUL byte among its events resolved so far (0: none), and either 0x80000000 | L when all its packets have L bytes or
//   (ke - ks) / (e_rel - b_rel) as a float (the interpolation guess of the packet lookup) --
// then, at byte 64, {parity of the item being scanned, how many of the pending events belong to items before it}, and at
// byte 72 the state of the warp's candidate ring (two words).
constexpr uint32_t SC_STATE = 64, SC_CAND = 72;

extern __shared__ __align__(1024) uint8_t smem[];
// shared address of the dynamic shared memory (uniform registers; the generic-to-shared conversion costs more)
__device__ __forceinline__ uint32_t smem_sa()
{
    uint32_t a;
    asm("mov.u32 %0, smem;" : "=r"(a));
    return a;
}
__device__ __forceinline__ uint32_t dc(uint32_t k) { return lds32(smem_sa() + UN_OFF_MISC + 4u * k); }
__device__ __forceinline__ const uint8_t *dc_ptr(uint32_t k)
{
    const uint2 v = lds64(smem_sa() + UN_OFF_MISC + 4u * k);
    return reinterpret_cast<const uint8_t *>(((uint64_t)v.y << 32) | v.x);
}
__device__ __forceinline__ uint32_t warp_q_sa() { return smem_sa() + UN_OFF_Q + (threadIdx.x >> 5) * (UN_QCAP * UN_Q_BYTES1); }
__device__ __forceinline__ uint32_t warp_t_sa() { return smem_sa() + UN_OFF_T + (threadIdx.x >> 5) * (UN_QDRAIN * UN_T_BYTES1); }
__device__ __forceinline__ uint32_t warp_scratch_sa() { return smem_sa() + UN_OFF_SCRATCH + (threadIdx.x >> 5) * 128; }

// what a resolve step needs besides the events; every warp derives it from its own index (nothing of it has to live in
// the row loop's registers)
struct drain_args {
    uint32_t q_sa;       // the warp's event ring
    uint32_t scratch_sa; // the warp's scratch words
    uint32_t vtab_sa;    // the probe tables in shared memory, 0 = in global memory
    uint32_t counts_sa;  // the shared counters, or 0
};

__device__ __forceinline__ void count_hit(const drain_args &d, uint32_t u)
{
    if (d.counts_sa) asm volatile("red.shared.add.u32 [%0], 1;" ::"r"(d.counts_sa + 4u * u) : "memory");
    else atomicAdd(reinterpret_cast<unsigned long long *>(const_cast<uint8_t *>(dc_ptr(DC_CNT_LO))) + u, 1ull);
}

// The find kernel's hit (after count_hit): one 16-byte record {absolute position, distinct id} that the locate kernel
// (find.cu) turns into {packet, offset, pattern}.  Slots are reserved by one atomic per group of lanes that hit
// together: a single counter takes every match of the batch (C3: 33.8 M per pass), one atomic per hit would serialise
// on it.  Every match is counted; those whose slot lies past the capacity are not written.
__device__ __forceinline__ void emit_hit(const uint64_t pos, const uint32_t u)
{
    namespace cg = cooperative_groups;
    const cg::coalesced_group g = cg::coalesced_threads();
    unsigned long long base = 0;
    if (g.thread_rank() == 0)
        base = atomicAdd(reinterpret_cast<unsigned long long *>(const_cast<uint8_t *>(dc_ptr(DC_FOUND_LO))), (unsigned long long)g.size());
    const uint64_t slot = g.shfl(base, 0) + g.thread_rank();
    const uint2 cap = lds64(smem_sa() + UN_OFF_MISC + 4u * DC_CAP_LO);
    if (slot < (((uint64_t)cap.y << 32) | cap.x)) {
        uint4 *rec = reinterpret_cast<uint4 *>(const_cast<uint8_t *>(dc_ptr(DC_REC_LO))) + slot;
        __stcs(rec, make_uint4((uint32_t)pos, (uint32_t)(pos >> 32), 0u, u));
    }
}
template <bool EMIT>
__device__ __forceinline__ void hit(const drain_args &d, const uint32_t u, const uint64_t pos)
{
    count_hit(d, u);
    if (EMIT) emit_hit(pos, u);
}

// 4 text bytes starting at g, of which the first `need` (>= 1) matter: never read past the word that holds the last
// needed byte, which lies inside the packet.
__device__ __forceinline__ uint32_t text_window(const uint8_t *g, uint32_t need)
{
    const uint32_t sh = (uint32_t)reinterpret_cast<uintptr_t>(g) & 3u;
    const uint32_t *gw = reinterpret_cast<const uint32_t *>(g - sh);
    const uint32_t lo = __ldg(gw);
    const uint32_t hi = sh + (need < 4 ? need : 4u) > 4u ? __ldg(gw + 1) : 0u;
    return __funnelshift_r(lo, hi, 8u * sh);
}

// where the probe tables' parts are, read once per resolve step
struct probe_consts {
    uint32_t slots_a, shift_a, slots_b, shift_b, one, rec;
};
// A candidate: text bytes 0..3 (x0) and 4..7 (x1) from its start, `room` (>= 1) = bytes from its start to the end of its
// packet, pos = its absolute position.  Every pattern that starts there and is at most `room` bytes long is counted.
// The candidate's first two bytes select one slot of probe table A (the two-byte patterns), its first three one slot of
// table B (the longer ones); the slots' records carry the pattern's first 8 bytes and their masks, so a record costs one
// 16-byte load and one masked compare, and only a record that agrees on those bytes is looked at further (patterns of
// more than 8 bytes: word by word against the text in global memory -- L2, the row was read a moment ago).
template <bool VS, bool EMIT>
__device__ __forceinline__ void verify_cand(const drain_args &d, const probe_consts &pc, const uint32_t x0, const uint32_t x1,
                                            const uint32_t room, const uint64_t pos)
{
    const uint32_t *vtab_g = VS ? nullptr : reinterpret_cast<const uint32_t *>(dc_ptr(DC_VTAB_LO));
    auto vt = [&](uint32_t word) -> uint32_t { return VS ? lds32(d.vtab_sa + 4u * word) : __ldg(vtab_g + word); };
    auto vt4 = [&](uint32_t word) -> uint4 {
        return VS ? lds128(d.vtab_sa + 4u * word) : __ldg(reinterpret_cast<const uint4 *>(vtab_g + word));
    };
    auto vt2 = [&](uint32_t word) -> uint2 {
        return VS ? lds64(d.vtab_sa + 4u * word) : __ldg(reinterpret_cast<const uint2 *>(vtab_g + word));
    };
    const uint32_t vt_one = pc.one, vt_slots_a = pc.slots_a, vt_slots_b = pc.slots_b;
    if (vt_one) { // one-byte patterns: a direct table (room >= 1 always holds)
        const uint32_t u = vt(vt_one + (x0 & 0xffu));
        if (u != 0xffffffffu) hit<EMIT>(d, u, pos);
    }
    if (room < 2) return;
    uint2 ea = make_uint2(0, 0), eb = make_uint2(0, 0); // {first record, records}
    if (vt_slots_a) ea = vt2(vt_slots_a + 2u * (((x0 & 0xffffu) * 0x9e3779b1u) >> pc.shift_a));
    if (vt_slots_b && room >= 3) eb = vt2(vt_slots_b + 2u * (((x0 & 0xffffffu) * 0x9e3779b1u) >> pc.shift_b));
    const uint32_t nrec = ea.y + eb.y;
    if (nrec == 0) return; // most candidates end here: no pattern begins with these bytes
    const uint32_t vt_rec = pc.rec;
    for (uint32_t j = 0; j < nrec; j++) {
        const uint32_t r = vt_rec + 8u * (j < ea.y ? ea.x + j : eb.x + (j - ea.y));
        const uint4 a = vt4(r); // pattern bytes 0..3, their mask, bytes 4..7, their mask
        if ((((x0 ^ a.x) & a.y) | ((x1 ^ a.z) & a.w)) != 0) continue;
        const uint2 b = vt2(r + 4); // length, distinct id
        const uint32_t m = b.x;
        // m <= room: else it would end past the packet (serial.c:191: the text ends there); the bytes of x0/x1 past
        // `room` are not text of this packet, but a pattern that short compares none of them
        if (m > room) continue;
        bool same = true;
        if (m > 8) {
            const uint32_t pw0 = dc(DC_BLOB) + vt(r + 6);
            const uint8_t *g = dc_ptr(DC_TEXT_LO) + pos;
            for (uint32_t jj = 8; jj < m && same; jj += 4) { // pattern bytes jj..jj+3 against text bytes jj..
                const uint32_t pw = vt(pw0 + (jj >> 2)), rem = m - jj;
                const uint32_t diff = text_window(g + jj, rem) ^ pw;
                same = (rem >= 4 ? diff : diff & ((1u << (8 * rem)) - 1u)) == 0;
            }
        }
        if (same) hit<EMIT>(d, b.y, pos);
    }
}

// The warp's candidate ring: what phase 1 of the resolve steps found alive waits here until 32 have come together, so
// that phase 2 always runs with every lane busy (the candidates of one resolve step seldom fill a whole number of
// rounds).  A slot: {x0, x1, position low word, room | position high bits << 8}.  State (scratch, SC_CAND): two
// free-running counters, slots handed out and slots verified.
__device__ __forceinline__ uint32_t warp_c_sa() { return smem_sa() + UN_OFF_C + (threadIdx.x >> 5) * (UN_CCAP * UN_C_BYTES1); }
// verify the n (<= 32) candidates from slot `head` on, one per lane
template <bool EMIT>
__device__ __forceinline__ void verify_round(const drain_args &d, const uint32_t head, const uint32_t n)
{
    const uint32_t lane = threadIdx.x & 31;
    if (lane < n) {
        probe_consts pc;
        const uint4 c0 = lds128(smem_sa() + UN_OFF_MISC + 4u * DC_SLOTS_A);
        const uint2 c1 = lds64(smem_sa() + UN_OFF_MISC + 4u * DC_ONE);
        pc.slots_a = c0.x; pc.shift_a = c0.y; pc.slots_b = c0.z; pc.shift_b = c0.w; pc.one = c1.x; pc.rec = c1.y;
        const uint4 e = lds128v(warp_c_sa() + ((head + lane) & (UN_CCAP - 1)) * UN_C_BYTES1);
        const uint64_t pos = ((uint64_t)(e.w >> 8) << 32) | e.z;
        if (d.vtab_sa) verify_cand<true, EMIT>(d, pc, e.x, e.y, e.w & 0xffu, pos);
        else verify_cand<false, EMIT>(d, pc, e.x, e.y, e.w & 0xffu, pos);
    }
}
// the candidates still waiting at the end of a batch
template <bool EMIT>
__device__ __forceinline__ void flush_body()
{
    drain_args d;
    d.q_sa = warp_q_sa();
    d.scratch_sa = warp_scratch_sa();
    d.vtab_sa = dc(DC_VTAB_SA);
    d.counts_sa = dc(DC_COUNTS_SA);
    __syncwarp();
    const uint2 cs = lds64v(d.scratch_sa + SC_CAND); // {handed out, verified}: fewer than 32 apart between resolve steps
    verify_round<EMIT>(d, cs.y, cs.x - cs.y);
    __syncwarp();
    if ((threadIdx.x & 31) == 0) sts32v(d.scratch_sa + SC_CAND + 4, cs.x);
    __syncwarp();
}
__device__ __noinline__ void flush_candidates() { flush_body<false>(); }
__device__ __noinline__ void flush_candidates_find() { flush_body<true>(); }

// Phase 0 of a resolve step, on its own so that the row loop can issue it a row or two ahead: the n (<= 32) oldest
// events' groups (32 B + 8 B lookahead), one per lane, from L2 (the rows were read a few microseconds ago) straight
// into the warp's staging slots.  The row loop stores 8 bytes per event instead of 48 and keeps no row in registers
// for it.  A group at or past its item's end reported from registers that were not loaded and holds nothing of the
// item: zeros.  cp.async: no registers, and nobody waits here.
__device__ __forceinline__ void drain_fetch(const uint32_t head, const uint32_t n)
{
    const uint32_t lane = threadIdx.x & 31;
    if (lane < n) {
        const uint2 t = lds64v(warp_q_sa() + ((head + lane) & (UN_QCAP - 1)) * UN_Q_BYTES1);
        const uint32_t tx = t.x;
        const uint32_t gq = (tx & 0x7fffffffu) << 5;
        const uint32_t set_sa = warp_scratch_sa() + ((tx >> 31) << 5); // the event's item
        const uint32_t e_rel = lds32v(set_sa + 12);
        const uint2 r0 = lds64v(set_sa + 16);
        // the lookahead matters to the last quarter's starts only (25..31: the re-run's bytes 32..35, a candidate's bytes
        // up to 38); an LDGSTS is charged by the lane, so the other events' lanes sit this one out
        const bool in = gq < e_rel, more = in && (t.y >> 24) != 0 && gq + UN_GRP < ((e_rel + 31u) & ~31u);
        const uint8_t *src = dc_ptr(DC_TEXT_LO) + (((uint64_t)r0.y << 32) | r0.x) + (in ? gq : 0u);
        const uint32_t dst = warp_t_sa() + lane * UN_T_BYTES1;
        cp_async16(dst, src, in ? 16u : 0u);
        cp_async16(dst + 16, src + 16, in ? 16u : 0u);
        if (more) cp_async8(dst + 32, src + 32, 8u);
    }
}

// Resolve the n (<= 32) oldest events of the warp's ring, which start at slot `head`.
//
// Phase 1, one event per lane: which start positions of the event's quarter(s) fired, where the NULs are, which
// packet(s) they lie in -> mask of candidate starts that are alive (inside the item, no NUL before them in their
// packet) and mask of packet boundaries inside the group.
// Phase 2: the alive candidates go to the warp's candidate ring; every 32 of them are verified, one per lane: probe,
// compare, count.
//
// The events belong to the work item the warp is scanning or to the one before it (the row loop sees to that); an
// event carries its item's parity, and what the resolve step has to know about either item waits in the warp's
// scratch words, where the warp put it when it took the item: no lane has to look anything up in global memory for
// it, and the row loop does not keep it in registers.  Positions are relative to the item's row0 (32 bits).
template <bool EMIT>
__device__ __forceinline__ void drain_body(const uint32_t head, const uint32_t n)
{
    drain_args d;
    d.q_sa = warp_q_sa();
    d.scratch_sa = warp_scratch_sa();
    d.vtab_sa = dc(DC_VTAB_SA);
    d.counts_sa = dc(DC_COUNTS_SA);
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t lutL = smem_sa() + (lane << 2), mul2 = dc(DC_MUL4096);
    uint32_t lt;
    asm("mov.u32 %0, %%lanemask_lt;" : "=r"(lt));
    cp_async_wait_all(); // phase 0 (drain_fetch): my event's bytes are in its slot
    __syncwarp();
    const uint32_t t_sa = warp_t_sa();
    const uint32_t entry_sa = t_sa + lane * UN_T_BYTES1; // my event's slot among the 32 being resolved
    uint32_t cm = 0, zm = 0, gq = 0, par = 0;
    uint32_t ks = 0, ke = 0, b_rel = 0, e_rel = 0, row0_lo = 0, row0_hi = 0, carry = 0, psize = 0;
    if (lane < n) {
        const uint2 t = lds64v(d.q_sa + ((head + lane) & (UN_QCAP - 1)) * UN_Q_BYTES1); // group index (relative to row0) | item parity << 31, quarter reports
        par = t.x >> 31;
        gq = (t.x & 0x7fffffffu) << 5;
        const uint32_t set_sa = d.scratch_sa + (par << 5); // my item's scratch set
        const uint4 s0 = lds128v(set_sa), s1 = lds128v(set_sa + 16);
        ks = s0.x; ke = s0.y; b_rel = s0.z; e_rel = s0.w;
        row0_lo = s1.x; row0_hi = s1.y; carry = s1.z; psize = s1.w;
        // Re-run the filter over the quarters that reported (usually one), one byte per update, this time recording
        // which start positions fired and which bytes are NUL.  Quarter k: bytes 8k..8k+11 -- three bytes of run-in,
        // then the starts 8k..8k+8 report at the bytes 8k+3..8k+11, and so do the NULs among the bytes 8k..8k+8 (the
        // quarters of the row loop overlap by one start; OR-ing a bit twice changes nothing).
        uint32_t quarters = (((t.y & 0x7f7f7f7fu) + 0x7f7f7f7fu) | t.y) & 0x80808080u; // bit 8k+7: quarter k
        while (quarters) {
            const uint32_t k8 = (__ffs(quarters) - 1) & ~7u; // 8k
            quarters &= quarters - 1;
            const uint2 w01 = lds64v(entry_sa + k8);
            const uint32_t w0 = w01.x, w1 = w01.y, w2 = lds32v(entry_sa + k8 + 8);
            uint32_t S = 0, cmr = 0, zr = 0;
            // Two bytes per update, as in the row loop; after an update bits 24..28 / 18..22 hold the candidate buckets of
            // the start three before b0 / b1, bits 29 / 23 "that byte is NUL".  Adding 0x1f to a 5-bit field carries into
            // the bit above it iff the field is not zero, and x * 132 moves bits 29 and 23 of x to bits 31 and 30: two
            // report bits per update and kind, shifted into cmr / zr from below (nothing can report before byte 3).
#define SV2(word, k0)                                                                                           \
    do {                                                                                                        \
        SA2(word, k0);                                                                                          \
        zr = __funnelshift_l((S & 0x20800000u) * 132u, zr, 2);                                                  \
        cmr = __funnelshift_l((((S & 0x1f7c0000u) + 0x1f7c0000u) & 0x20800000u) * 132u, cmr, 2);               \
    } while (0)
            SA2(w0, 0);
            SV2(w0, 2);
            SV2(w1, 0); SV2(w1, 2);
            SV2(w2, 0); SV2(w2, 2);
#undef SV2
            cm |= (__brev(cmr) >> 23) << k8; // the first report is the highest of the 9 bits
            zm |= (__brev(zr) >> 23) << k8;
        }
        // the item's first and last rows overhang it: starts count inside [b_rel, e_rel) only, and bytes
        // past e_rel may be anything, so NULs count below e_rel only
        const uint32_t lo = clamp32((int32_t)b_rel - (int32_t)gq), hi = clamp32((int32_t)e_rel - (int32_t)gq);
        cm &= bit_window(lo, hi);
        zm &= bits_below(hi);
    }
    // last NUL before my event's bytes: the nearest earlier event of the same item that holds one, else the carry of
    // my item (the events of an item are in stream order; those of the older item come first)
    const uint32_t mylast1 = zm ? gq + (32u - __clz(zm)) : 0u; // 1 + position of my last NUL
    const uint32_t nulm = __ballot_sync(FULL, zm != 0), parm = __ballot_sync(FULL, par != 0);
    const uint32_t mine = nulm & (par ? parm : ~parm);
    const uint32_t below = mine & lt;
    const uint32_t from_below = __shfl_sync(FULL, mylast1, below ? 31 - __clz(below) : 0);
    const uint32_t prev1 = below ? from_below : carry;
    // the carries: the last NUL of either item among these events is stored by the lane that holds it -- the one with
    // a NUL and no lane of its item with a NUL above it
    uint32_t gt;
    asm("mov.u32 %0, %%lanemask_gt;" : "=r"(gt));
    __syncwarp();
    if (zm && !(mine & gt)) sts32v(d.scratch_sa + (par << 5) + 24, mylast1);

    uint32_t am = 0, bm = 0, nextb = 255; // alive candidates; packet starts inside the group (bit = offset);
                                          // offset of the first packet start at or after the group's end
    if (cm) {
        // The packet that holds my first candidate: the last k in [ks, ke) with offsets[k] <= p0.  When all the item's
        // packets have the same size (the row loop found out when it took the item) it is a division; otherwise a guess
        // by interpolation, then a binary search in what is left of the item's slice of `offsets` (relative to row0 they
        // fit 32 bits and need the low words only).
        const uint32_t p0 = gq + (__ffs(cm) - 1);
        const bool uniform = (psize >> 31) != 0;
        const uint32_t L = psize & 0x7fffffffu;
        const uint32_t *olo = reinterpret_cast<const uint32_t *>(dc_ptr(DC_OFF_LO));
        auto orel = [&](uint32_t k) -> uint32_t { return __ldg(olo + 2u * k) - row0_lo; };
        uint32_t k, ps, pe;
        if (uniform) {
            const uint32_t x = p0 - b_rel;
            // (1 / L waits in the set's first word -- a uniform item has no use for its first packet's index)
            const uint32_t q = (uint32_t)((float)x * __uint_as_float(ks)); // x < 2^24 or the quotient is small: off by one at most
            int32_t r = (int32_t)(x - q * L);
            if (r < 0) r += (int32_t)L;
            if (r >= (int32_t)L) r -= (int32_t)L;
            k = 0;
            ps = p0 - (uint32_t)r;
            pe = ps + L;
        } else {
            uint32_t k1 = ke;
            k = ks;
            uint32_t kg = ks + (uint32_t)((float)(p0 - b_rel) * __uint_as_float(psize));
            kg = kg >= ke ? ke - 1 : kg;
            const uint32_t o0 = orel(kg), o1 = orel(kg + 1);
            if (o0 <= p0) {
                k = kg;
                if (p0 < o1) k1 = kg + 1;
                else k = kg + 1; // offsets[kg + 1] <= p0 < e_rel, so kg + 1 < ke
            } else {
                k1 = kg;
            }
            while (k1 - k > 1) {
                const uint32_t mid = k + (k1 - k) / 2;
                if (orel(mid) <= p0) k = mid; else k1 = mid;
            }
            ps = orel(k);
            pe = orel(k + 1);
        }
        bool dead = prev1 > ps; // a NUL in [ps, my bytes): kmp_matcher's strlen() stopped before them
        uint32_t a = ps > gq ? ps - gq : 0u; // the packet [ps, pe) covers my group from offset a on
        for (;;) {
            const uint32_t b = pe - gq >= 32 ? 32u : pe - gq;
            const uint32_t seg = bit_window(a, b), z = zm & seg;
            if (!dead) am |= cm & seg & (z ? (z & (0u - z)) - 1u : FULL); // starts before the packet's first NUL
            if (b == 32) break;
            bm |= 1u << b;          // the next packet starts inside my group
            if (pe >= e_rel) break; // ... or the item ends there (what may follow are empty packets): nothing beyond is mine
            a = b;
            dead = false;
            k++;
            ps = pe;
            pe = uniform ? pe + L : orel(k + 1);
        }
        nextb = pe - gq > 255 ? 255u : pe - gq;
    }
    // Phase 2.  Every lane appends its alive candidates to the warp's candidate ring, and whenever 32 are waiting they are
    // verified, one per lane -- whichever event they came from, this resolve step's or an earlier one's.  (A candidate is
    // self-contained: its first 8 bytes, its position, the bytes left in its packet.)
    const uint64_t gpos = (((uint64_t)row0_hi << 32) | row0_lo) + gq; // absolute position of my group (a multiple of 32)
    const uint32_t gpos_lo = (uint32_t)gpos, gpos_hi8 = (uint32_t)(gpos >> 32) << 8;
    const uint32_t c_sa = warp_c_sa(), cst_sa = d.scratch_sa + SC_CAND;
    const bool walls = __any_sync(FULL, bm != 0); // some group of this step holds a packet boundary (C3: one step in two)
    // my first alive candidate goes to `slot`
    auto push_one = [&](const uint32_t slot) {
        const uint32_t i = __ffs(am) - 1;
        am &= am - 1;
        const uint32_t a = entry_sa + (i & ~3u), sh = 8u * (i & 3u);
        const uint32_t w0 = lds32v(a), w1 = lds32v(a + 4), w2 = lds32v(a + 8); // i + 7 < 40: inside the event's text
        uint32_t end = nextb; // the end of the candidate's packet: the first packet start after byte i
        if (walls) {
            const uint32_t above = bm & ~((2u << i) - 1u);
            if (above) end = (uint32_t)__ffs(above) - 1u;
        }
        sts128v(c_sa + (slot & (UN_CCAP - 1)) * UN_C_BYTES1, __funnelshift_r(w0, w1, sh), __funnelshift_r(w1, w2, sh),
                gpos_lo | i, (end - i) | gpos_hi8);
    };
    const uint2 cs0 = lds64v(cst_sa); // {slots handed out, slots verified}; fewer than 32 candidates are waiting
    uint32_t ctail = cs0.x, chead = cs0.y;
    // every lane's run of slots: a prefix sum of the counts (a shared-memory atomic would serialise its 20-odd lanes on
    // the pipe the filter's lookups need)
    const uint32_t cnt = __popc(am);
    uint32_t incl = cnt;
#pragma unroll
    for (uint32_t dd = 1; dd < 32; dd <<= 1)
        asm volatile("{\n\t.reg .pred p;\n\t.reg .b32 v;\n\t"
                     "shfl.sync.up.b32 v|p, %0, %1, 0, 0xffffffff;\n\t"
                     "@p add.u32 %0, %0, v;\n\t}"
                     : "+r"(incl)
                     : "r"(dd));
    const uint32_t total = __shfl_sync(FULL, incl, 31);
    if (ctail - chead + total <= UN_CCAP) {
        // The ring takes them all: every lane fills its run at its own pace -- no trips in step with the lane that has
        // the most.  (The order of the candidates in the ring does not matter.)
        uint32_t slot = ctail + incl - cnt;
        while (am) push_one(slot++);
        ctail += total;
        __syncwarp();
    } else {
        // (dense candidates: trips of at most one candidate per lane, verified as soon as 32 are waiting)
        for (;;) {
            const uint32_t any = __ballot_sync(FULL, am != 0);
            if (any == 0) break;
            if (am) push_one(ctail + __popc(any & lt));
            ctail += __popc(any);
            __syncwarp();
            if (ctail - chead >= 32u) {
                verify_round<EMIT>(d, chead, 32u);
                chead += 32u;
                __syncwarp();
            }
        }
    }
    while (ctail - chead >= 32u) {
        verify_round<EMIT>(d, chead, 32u);
        chead += 32u;
    }
    __syncwarp();
    if (lane == 0) sts64v(cst_sa, ctail, chead);
    __syncwarp();
}

// the same out of line, for the places that are not in the row loop (taking an item, the end of the batch): a call in
// the row loop itself would cost that loop five spilled registers (the callee's needs bind at every call site)
__device__ __noinline__ void drain_events(const uint32_t head, const uint32_t n)
{
    drain_fetch(head, n);
    drain_body<false>(head, n);
}
__device__ __noinline__ void drain_events_find(const uint32_t head, const uint32_t n)
{
    drain_fetch(head, n);
    drain_body<true>(head, n);
}

// NUL-dense row.  An event without candidates exists only to tell later candidates where the last NUL before them
// is; when the next event of the row is of the same kind, that one tells them a later NUL and this one is not needed:
// its reports are cleared (binary payloads: one event per row instead of one per group).  m = lanes with reports,
// has_cand = my reports hold a candidate.  Kept out of line: the row loop should stay small.
__device__ __noinline__ uint32_t drop_superseded(uint32_t tops, const uint32_t m, const bool has_cand)
{
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t mc = __ballot_sync(FULL, has_cand);                  // lanes with candidates
    const uint32_t above = m & ~((2u << lane) - 1u);                    // reporting lanes above me
    if (!((mc >> lane) & 1u) && above && !((mc >> (__ffs(above) - 1)) & 1u)) tops = 0;
    return tops;
}

// warp-uniform value, in a form the compiler can keep in a uniform register
__device__ __forceinline__ uint32_t uni(uint32_t v) { return __shfl_sync(FULL, v, 0); }
__device__ __forceinline__ uint64_t uni(uint64_t v) { return __shfl_sync(FULL, v, 0); }
#undef DP_SEL
#define DP_SEL(k) p.sel[k]
// The kernel body, in two instantiations: the count kernel (EMIT = false) and the find kernel (EMIT = true), which
// also writes a record per match; what it needs of the record buffer waits in the DC_* words, not in registers.
template <bool EMIT>
__device__ __forceinline__ void union_body(const union_params &__restrict__ p, const kmpb_find_out &__restrict__ fo)
{
    uint32_t *lut = reinterpret_cast<uint32_t *>(smem);                      // L, then G
    uint32_t *s_misc = reinterpret_cast<uint32_t *>(smem + UN_OFF_MISC);
    uint32_t *s_counts = reinterpret_cast<uint32_t *>(smem + UN_OFF_COUNTS);
    const uint32_t n_uniq = p.n_uniq; // read unconditionally: p is a reference here, a load under the condition would branch
    const uint32_t counts_bytes = p.counts_in_smem ? ((4u * n_uniq + 15u) & ~15u) : 0u;
    uint32_t *s_vtab = reinterpret_cast<uint32_t *>(smem + UN_OFF_COUNTS + counts_bytes);

    for (uint32_t i = threadIdx.x; i < 256 * 32; i += UN_THREADS) {
        const uint32_t f = p.filter[i >> 5];
        lut[i] = f;                                // L[c] for lane i & 31
        lut[256 * 32 + i] = (f << 6) | 0x3fu;      // G[c]
    }
    if (p.counts_in_smem)
        for (uint32_t i = threadIdx.x; i < p.n_uniq; i += UN_THREADS) s_counts[i] = 0;
    if (p.vtab_in_smem)
        for (uint32_t i = threadIdx.x; i < p.vtab_words; i += UN_THREADS) s_vtab[i] = p.vtab[i];
    for (uint32_t i = threadIdx.x; i < UN_SCRATCH_BYTES / 4; i += UN_THREADS)
        reinterpret_cast<uint32_t *>(smem + UN_OFF_SCRATCH)[i] = 0; // item parity, pending flag, carries
    if (threadIdx.x == 0) {
        const uint64_t text0 = reinterpret_cast<uint64_t>(p.bytes) - p.abs_base, off = reinterpret_cast<uint64_t>(p.offsets);
        const uint64_t vt = reinterpret_cast<uint64_t>(p.vtab), cn = reinterpret_cast<uint64_t>(p.uniq_counts);
        s_misc[DC_TEXT_LO] = (uint32_t)text0; s_misc[DC_TEXT_HI] = (uint32_t)(text0 >> 32);
        s_misc[DC_OFF_LO] = (uint32_t)off; s_misc[DC_OFF_HI] = (uint32_t)(off >> 32);
        s_misc[DC_VTAB_LO] = (uint32_t)vt; s_misc[DC_VTAB_HI] = (uint32_t)(vt >> 32);
        s_misc[DC_CNT_LO] = (uint32_t)cn; s_misc[DC_CNT_HI] = (uint32_t)(cn >> 32);
        s_misc[DC_SLOTS_A] = p.vt_slots_a; s_misc[DC_SHIFT_A] = p.vt_shift_a;
        s_misc[DC_SLOTS_B] = p.vt_slots_b; s_misc[DC_SHIFT_B] = p.vt_shift_b;
        s_misc[DC_ONE] = p.vt_one; s_misc[DC_REC] = p.vt_rec; s_misc[DC_BLOB] = p.vt_blob;
        s_misc[DC_MUL4096] = p.mul4096;
        s_misc[DC_VTAB_SA] = p.vtab_in_smem ? saddr_of(s_vtab) : 0u;
        s_misc[DC_COUNTS_SA] = p.counts_in_smem ? saddr_of(s_counts) : 0u;
        if (EMIT) {
            const uint64_t rec = reinterpret_cast<uint64_t>(fo.rec), found = reinterpret_cast<uint64_t>(fo.found);
            s_misc[DC_REC_LO] = (uint32_t)rec; s_misc[DC_REC_HI] = (uint32_t)(rec >> 32);
            s_misc[DC_CAP_LO] = (uint32_t)fo.capacity; s_misc[DC_CAP_HI] = (uint32_t)(fo.capacity >> 32);
            s_misc[DC_FOUND_LO] = (uint32_t)found; s_misc[DC_FOUND_HI] = (uint32_t)(found >> 32);
        }
    }
    const uint32_t lane = threadIdx.x & 31;
    __syncthreads();

        static_assert(UN_LUT_BYTES == 32768, "lds32_g's immediate offset");
    uint32_t lutL = smem_sa() + (lane << 2); // L starts the dynamic shared memory
    asm volatile("" : "+r"(lutL));             // opaque: a value to keep in its register, not an expression to recompute
    const uint32_t mul2 = p.mul4096;
    const uint32_t q_sa = warp_q_sa();
    // The event ring's state in one register: byte offset in the ring of the slot the next event goes to << 22 | pending
    // events.  The ring is 2^10 bytes, so the offset wraps by falling off the top of the word (however many events a
    // warp sees in a launch) and an address is ring + (state >> 22); the oldest pending event sits `pending` slots
    // before the next one.
    static_assert(UN_QCAP * UN_Q_BYTES1 == 1024, "the ring offset lives in the top 10 bits of qs");
    static_assert(UN_QCAP == 128 && 2 * UN_QDRAIN + 2 * 32 <= UN_QCAP, "pending events fit 7 bits and the ring");
    // bit 8: the text of the 32 oldest events is on its way into the staging slots (drain_fetch was issued)
    constexpr uint32_t QS_SLOT = UN_Q_BYTES1 << 22, QS_PENDING = 0xffu, QS_FETCHED = 0x100u;
    uint32_t qs = 0;
    auto pending = [&]() -> uint32_t { return qs & QS_PENDING; };
    auto oldest = [&]() -> uint32_t { return ((qs >> 22) / UN_Q_BYTES1 - pending()) & (UN_QCAP - 1); };

    // resolve the oldest min(pending, 32) events (out of line: the rare places)
    auto resolve_oldest = [&]() {
        const uint32_t qn = pending(), n = qn < UN_QDRAIN ? qn : UN_QDRAIN;
        if (EMIT) drain_events_find(oldest(), n);
        else drain_events(oldest(), n);
        qs -= n;
    };

    for (;;) {
        uint32_t item = 0;
        if (lane == 0) item = atomicAdd(&p.work[0], 1u);
        item = uni(item);
        if (item >= p.n_items) break;
        const uint32_t ks = uni(p.items[item]), ke = uni(p.items[item + 1]);
        if (ks >= ke) continue;
        const uint64_t b_abs = uni(p.offsets[ks]), e_abs = uni(p.offsets[ke]);
        if (b_abs == e_abs) continue;
        if (e_abs - b_abs >= (1ull << 31) - 4096) { // only past KMPB_PACKET_LIMIT (the partition has flagged the packet)
            if (lane == 0) atomicOr(&p.work[1], 1u);
            continue;
        }
        // What the resolve step needs to know about this item goes into the scratch set of the item's parity.  The
        // set still belongs to the item before the previous one; its events are gone unless the list has not been
        // resolved since then (the flag: "the list holds events of the item before the one being scanned"), in
        // which case they are now.
        const uint2 st = lds64v(warp_scratch_sa() + SC_STATE); // parity of the previous item, pending events older than it
        const uint32_t par = st.x ^ 1u;
        if (st.y) // (the row loop counts them down as it resolves; an item of many rows leaves none)
            while (pending()) resolve_oldest();
        __syncwarp();
        const uint64_t row0 = b_abs & ~127ull; // absolute position of the item's first row
        const uint32_t b_rel = (uint32_t)(b_abs - row0), e_rel = (uint32_t)(e_abs - row0);
        // do all the item's packets have the same size?  (fixed-size records: the packet lookup becomes a division)
        uint32_t psize, word0 = ks;
        {
            const uint64_t L = uni(p.offsets[ks + 1]) - b_abs;
            bool same = L != 0 && L * (ke - ks) == e_abs - b_abs;
            for (uint32_t j = lane + 1; same && j < ke - ks; j += 32) same = p.offsets[ks + j] == b_abs + j * L;
            same = __all_sync(FULL, same);
            psize = same ? 0x80000000u | (uint32_t)L : __float_as_uint((float)(ke - ks) / (float)(e_rel - b_rel));
            if (same) word0 = __float_as_uint(__frcp_rn((float)(uint32_t)L)); // the packet lookup of such an item is a multiplication
        }
        if (lane == 0) {
            const uint32_t set_sa = warp_scratch_sa() + (par << 5);
            sts128v(set_sa, word0, ke, b_rel, e_rel);
            sts128v(set_sa + 16, (uint32_t)row0, (uint32_t)(row0 >> 32), 0u, psize);
            sts64v(warp_scratch_sa() + SC_STATE, par, pending());
        }
        // The loop state of a lane, kept small (the filter needs the registers):
        //   src  = its 32 bytes of the row being scanned,
        //   left = bytes from there to the end of what the item lets it load (<= 0: nothing of this row is its to load),
        //   gcur = its group's index relative to row0 (32-byte units) | the item's parity << 31.
        const uint8_t *src = p.bytes + (row0 - p.abs_base) + lane * UN_GRP;
        const uint32_t load_end = (e_rel + 31u) & ~31u; // readable: the batch up to its end rounded up to 32 (kmpb200.h)
        int32_t left = (int32_t)load_end - (int32_t)(lane * UN_GRP);
        uint32_t gcur = lane | par << 31;

        // The row `ahead` rows after the one being scanned, global -> registers: every lane its own 32 bytes with one
        // 256-bit load.  A lane whose group lies past what the item lets it load (rows past the item's end, the lanes
        // past load_end in its last row) loads the item's last group instead (src + left is load_end, whichever row
        // src is in): whatever it reports from that is cut to the item's byte range by the resolve step.  The L2
        // prefetch of the row UN_PF rows further on rides on the same address.
        auto load_row = [&](auto ahead_c, row_regs &b) {
            constexpr uint32_t ahead = decltype(ahead_c)::value;
            ldg256(b, src + (ptrdiff_t)min((int32_t)(ahead * UN_ROW), left - (int32_t)UN_GRP));
            if (UN_PF) prefetch_l2_if<(ahead + UN_PF) * UN_ROW>(left > (int32_t)((ahead + UN_PF) * UN_ROW), src);
        };

        // one row: filter its bytes, append the events, refill the buffer with the row UN_NBUF ahead, and resolve
        // 32 events once the list holds that many
        auto scan_row = [&](row_regs &b, row_regs &freed) {
            // the 4 bytes after my group: the next lane's first word; for lane 31 the first word of the next row, asked
            // for now (the row's own load is already on its way, so it comes from L2 or rides on that fill) and used last
            uint32_t la;
            asm volatile("{\n\t.reg .pred p, q;\n\t"
                         "shfl.sync.down.b32 %0|p, %1, 1, 0x1f, 0xffffffff;\n\t" // p: there is a lane above me
                         "setp.gt.and.s32 q, %2, 32, !p;\n\t"
                         "@q ld.global.L1::no_allocate.u32 %0, [%3+32];\n\t}"
                         : "=&r"(la)
                         : "r"(b.w[0]), "r"(left), "l"(src));
            // The buffer scanned before this one is free: the row UN_NBUF - 1 ahead goes into it -- NOW, after this row's
            // first use has waited for its own load, not at the end of the previous scan: ptxas tracks all the row loads
            // with one scoreboard, and a wait on it waits for every load issued so far (the first use of each row used
            // to wait for the load issued a few instructions before it: no prefetch distance at all).
            load_row(std::integral_constant<uint32_t, UN_NBUF - 1>{}, freed);

            // ---- shift-and filter over 36 bytes, two per update ---------------------------------------
            // Update j takes bytes 2j, 2j+1 and reports what starts at 2j-3 (bits 24..29) and 2j-2 (bits 18..23): the
            // bytes' candidate buckets and "this byte is NUL".  acc[k] collects the starts 0..8, 9..16, 17..24, 25..31.
            uint32_t S = 0, acc0, acc1, acc2, acc3;
            SA2(b.w[0], 0);                         // bytes 0, 1: nothing can report yet
            acc0 = SA2(b.w[0], 2);                  // starts -1 (nothing), 0
            acc0 |= SA2(b.w[1], 0);
            acc0 |= SA2(b.w[1], 2);
            acc0 |= SA2(b.w[2], 0);
            acc0 |= SA2(b.w[2], 2);                 // 7, 8
            acc1 = SA2(b.w[3], 0);                  // 9, 10
            acc1 |= SA2(b.w[3], 2);
            acc1 |= SA2(b.w[4], 0);
            acc1 |= SA2(b.w[4], 2);                 // 15, 16
            acc2 = SA2(b.w[5], 0);                  // 17, 18
            acc2 |= SA2(b.w[5], 2);
            acc2 |= SA2(b.w[6], 0);
            acc2 |= SA2(b.w[6], 2);                 // 23, 24
            acc3 = SA2(b.w[7], 0);                  // 25, 26
            acc3 |= SA2(b.w[7], 2);
            acc3 |= SA2(la, 0);                     // 29, 30
            S = (S * mul2 + 4095u) & LUT_G(la, 2);  // 31 (start 32 is the next lane's: no lookup for the second byte)
            acc3 |= S & F6_HI;
            // The reports of quarter k: byte 3 of acc[k] (b0's, bits 0..5) and byte 2 (b1's, bits 2..7), the four
            // quarters side by side; quarter k has something to resolve iff byte k of `tops` is nonzero.
            const uint32_t t3 = __byte_perm(__byte_perm(acc0, acc1, 0x0073), __byte_perm(acc2, acc3, 0x0073), 0x5410);
            const uint32_t t2 = __byte_perm(__byte_perm(acc0, acc1, 0x0062), __byte_perm(acc2, acc3, 0x0062), 0x5410);
            const uint32_t tops = (t2 & 0xfcfcfcfcu) | t3;
            const uint32_t m = __ballot_sync(FULL, tops != 0);

#ifdef KMPB_ABLATE_SLOW_PATH // measurement only (wrong counts): how fast is the fast path alone?
            if (m == 0x12345678u)
#endif
            {   // (no test for "no reports at all": one row in 500)
                uint32_t tp = tops, mp = m, n = __popc(m);
                if (UN_DENSE <= 32 && n >= UN_DENSE) {
                    // NUL-dense row: superseded NUL-only events are dropped first (a rare path of its own)
                    tp = drop_superseded(tops, m, ((t2 & 0x7c7c7c7cu) | (t3 & 0x1f1f1f1fu)) != 0);
                    mp = __ballot_sync(FULL, tp != 0);
                    n = __popc(mp);
                }
                // the ring takes it: fewer than 32 events were pending at the top of the loop, a row appends at most 32
                if (tp != 0) {
                    uint32_t lt;
                    asm("mov.u32 %0, %%lanemask_lt;" : "=r"(lt));
                    sts64v(q_sa + ((qs + __popc(mp & lt) * QS_SLOT) >> 22), gcur, tp); // where and what; the resolve step fetches the bytes
                }
                qs += n * (QS_SLOT + 1u);
            }
        };

        // the first UN_PF rows' lines: 128 bytes per lane and step
        if (UN_PF)
            for (uint32_t x = lane * 128u; x < UN_PF * UN_ROW; x += 4096u) prefetch_l2_if(x < load_end, src - lane * UN_GRP + x);
        // UN_NBUF rows per trip: the buffers are compile-time registers, no moves between them
        // (the last buffer gets its first row from the first scan)
        row_regs b0 = {}, b1 = {};
        load_row(std::integral_constant<uint32_t, 0>{}, b0);
#if KMPB_UN_NBUF >= 3
        row_regs b2 = {};
        load_row(std::integral_constant<uint32_t, 1>{}, b1);
#endif
#if KMPB_UN_NBUF >= 4
        row_regs b3 = {};
        load_row(std::integral_constant<uint32_t, 2>{}, b2);
#endif
        // next row; the item is through when lane 0 has nothing left (its rows start at multiples of 32)
        auto advance = [&]() -> bool {
            src += UN_ROW;
            left -= (int32_t)UN_ROW;
            gcur += UN_ROW / UN_GRP;
            // left + 32 * lane <= 0, with 32 * lane = 8 * (lutL - start of L): no lane index to recompute
            return (left >> 3) + (int32_t)(lutL - smem_sa()) <= 0;
        };
#pragma unroll 1
        for (;;) {
            // With the loads of the next two rows on their way: resolve the 32 oldest events if their text was asked
            // for a trip ago (or if the ring would not take two more rows otherwise) -- here and nowhere else in the
            // loop, inlined (one copy of the code, and no call whose register needs the loop would have to respect).
            while ((qs & QS_FETCHED) || pending() >= 2 * UN_QDRAIN) {
                if (!(qs & QS_FETCHED)) drain_fetch(oldest(), UN_QDRAIN);
                drain_body<EMIT>(oldest(), UN_QDRAIN);
                qs = (qs & ~QS_FETCHED) - UN_QDRAIN;
                if (lane == 0) { // that many fewer events of older items
                    const uint32_t older = lds32v(warp_scratch_sa() + SC_STATE + 4);
                    sts32v(warp_scratch_sa() + SC_STATE + 4, older > UN_QDRAIN ? older - UN_QDRAIN : 0u);
                }
            }
            // 32 or more pending: their text starts its way from L2 now and is resolved at the top of the next trip
            if (pending() >= UN_QDRAIN) {
                drain_fetch(oldest(), UN_QDRAIN);
                qs |= QS_FETCHED;
            }
#if KMPB_UN_NBUF == 2
            scan_row(b0, b1);
            if (advance()) break;
            scan_row(b1, b0);
            if (advance()) break;
#elif KMPB_UN_NBUF == 3
            scan_row(b0, b2);
            if (advance()) break;
            scan_row(b1, b0);
            if (advance()) break;
            scan_row(b2, b1);
            if (advance()) break;
#else
            scan_row(b0, b3);
            if (advance()) break;
            scan_row(b1, b0);
            if (advance()) break;
            scan_row(b2, b1);
            if (advance()) break;
            scan_row(b3, b2);
            if (advance()) break;
#endif
        }
        qs &= ~QS_FETCHED; // whoever resolves those events next asks for their text again
    }
    // leftovers
    while (pending()) resolve_oldest();
    if (EMIT) flush_candidates_find();
    else flush_candidates();

    __syncthreads();
    if (p.counts_in_smem)
        for (uint32_t u = threadIdx.x; u < p.n_uniq; u += UN_THREADS)
            if (s_counts[u]) atomicAdd(p.uniq_counts + u, (unsigned long long)s_counts[u]);

    // The merge of the partial counts (openmp_data.c:169-173) and, across GPUs, the MPI_Reduce(SUM) of
    // mpi_dumping.c:202, inside this kernel: the last block to arrive expands the distinct-pattern totals
    // to file order and adds them to every count vector it was given -- system-scope atomics, so a vector
    // may live in a peer GPU's memory.
    if (p.n_out) {
        __threadfence();
        __syncthreads();
        if (threadIdx.x == 0) s_misc[DC_LAST] = atomicAdd(&p.work[2], 1u) == gridDim.x - 1 ? 1u : 0u;
        __syncthreads();
        if (s_misc[DC_LAST]) {
            __threadfence();
            for (uint32_t i = threadIdx.x; i < p.n_pat; i += UN_THREADS) {
                const unsigned long long v = __ldcg(p.uniq_counts + p.pat_to_uniq[i]);
                if (v)
                    for (uint32_t r = 0; r < p.n_out; r++) atomicAdd_system(p.out[r] + i, v);
            }
        }
    }
}

__global__ void __launch_bounds__(UN_THREADS, 1) kmpb_union_kernel(const __grid_constant__ union_params p)
{
    union_body<false>(p, kmpb_find_out());
}

__global__ void __launch_bounds__(UN_THREADS, 1) kmpb_union_find_kernel(const __grid_constant__ union_params p,
                                                                        const __grid_constant__ kmpb_find_out fo)
{
    union_body<true>(p, fo);
}

// ---- host side ------------------------------------------------------------------------------------

// scratch for batches of up to max_batch_bytes: work counters and the item table, one set per slot
int kmpb_union_scratch(kmpb_ctx *ctx, uint64_t max_batch_bytes)
{
    size_t need = (size_t)(max_batch_bytes / UN_ITEM_BYTES) + UN_TAIL_ITEMS + 8;
    if (need <= ctx->items_cap && ctx->d_items && ctx->d_work) return KMPB_OK;
    cudaFree(ctx->d_items);
    ctx->d_items = nullptr;
    ctx->items_cap = 0;
    if (!ctx->d_work) {
        KMPB_CUDA(cudaMalloc((void **)&ctx->d_work, KMPB_COPY_STREAMS * 4 * sizeof(uint32_t)));
        KMPB_CUDA(cudaMemset(ctx->d_work, 0, KMPB_COPY_STREAMS * 4 * sizeof(uint32_t))); // no error flags yet
    }
    KMPB_CUDA(cudaMalloc((void **)&ctx->d_items, (size_t)KMPB_COPY_STREAMS * need * sizeof(uint32_t)));
    ctx->items_cap = need;
    return KMPB_OK;
}

int kmpb_launch_union(kmpb_ctx *ctx, const kmpb_batch &b, int slot, uint64_t *d_uniq_counts, cudaStream_t stream,
                      const kmpb_fused_out &out, const kmpb_find_out *find)
{
    const kmpb_tables &h = ctx->host;
    if (h.n_uniq == 0 || b.n_packets == 0 || b.end_byte == b.first_byte) return KMPB_OK;
    if (b.n_packets >= (1ull << 31)) return kmpb_fail(KMPB_ELIMIT, "more than 2^31-1 packets in one batch");
    if ((b.abs_base & 511) || ((uintptr_t)b.d_bytes & 31))
        return kmpb_fail(KMPB_EINVAL, "payload buffer must be 32-byte aligned");
    if (b.end_byte >= (1ull << 56)) // a candidate's absolute position travels in 56 bits
        return kmpb_fail(KMPB_ELIMIT, "absolute stream offsets of 2^56 and more");
    if (b.end_byte - b.abs_base >= (1ull << 36))
        return kmpb_fail(KMPB_ELIMIT, "more than 64 GiB of payload in one batch");
    const uint64_t span = b.end_byte - b.first_byte;
    // Taking an item costs a warp three dependent trips to L2 (ticket, item table, offsets); large batches
    // afford larger items (C3, 14 GB: 64 KB items 2.96 TB/s, 256 KB items 3.00 TB/s).
    const uint64_t item_bytes = span >= (8ull << 30) ? 4ull * UN_ITEM_BYTES : span >= (4ull << 30) ? 2ull * UN_ITEM_BYTES : UN_ITEM_BYTES;
    // full-size items, except the last UN_TAIL_ITEMS small items (at most an eighth of the batch), so that the warps
    // run dry within a few rows of each other at the end of the batch: an eighth of a full item, at least 16 KB
    // (C3 with 256 KB items: 64 KB tails 3003 GB/s, 32 KB 3013, 16 KB 2995, 8 KB 2985)
    const uint64_t tail_div = std::min<uint64_t>(8, item_bytes / (UN_ITEM_BYTES / 4));
    const uint64_t whole = span / item_bytes;
    const uint64_t small_bytes = item_bytes / tail_div;
    const uint64_t tail_items = std::min<uint64_t>(UN_TAIL_ITEMS / tail_div, whole / 8); // at most an eighth of the batch
    const uint32_t n_big = (uint32_t)(whole - tail_items);
    const uint64_t small_span = span - (uint64_t)n_big * item_bytes;
    const uint32_t n_items = n_big + (uint32_t)((small_span + small_bytes - 1) / small_bytes);
    if ((size_t)n_items + 1 > ctx->items_cap) return kmpb_fail(KMPB_ESTATE, "union scratch too small");
    uint32_t *d_items = ctx->d_items + (size_t)slot * ctx->items_cap;
    uint32_t *d_work = ctx->d_work + slot * 4;

    // the counters and the probe tables go into shared memory if the block's 227 KB allow it
    const bool counts_in_smem = UN_SMEM_FIXED + 4ull * h.n_uniq + 16 <= UN_SMEM_MAX - 8192;
    const size_t counts_bytes = counts_in_smem ? ((4ull * h.n_uniq + 15) & ~15ull) : 0;
    const bool vtab_in_smem = UN_SMEM_FIXED + counts_bytes + 4ull * h.vtab_words <= UN_SMEM_MAX;
    const size_t smem_bytes = UN_SMEM_FIXED + counts_bytes + (vtab_in_smem ? 4ull * h.vtab_words : 0);
    if (!ctx->attr_union_set) {
        KMPB_CUDA(cudaFuncSetAttribute(kmpb_union_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)UN_SMEM_MAX));
        KMPB_CUDA(cudaFuncSetAttribute(kmpb_union_find_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)UN_SMEM_MAX));
        ctx->attr_union_set = true;
    }
    kmpb_union_partition_kernel<<<(n_items + 1 + 255) / 256, 256, 0, stream>>>(b.d_offsets, (uint32_t)b.n_packets, n_items,
                                                                              n_big, item_bytes, small_bytes, d_items, d_work);
    union_params p;
    p.bytes = b.d_bytes;
    p.abs_base = b.abs_base;
    p.offsets = b.d_offsets;
    p.n_packets = (uint32_t)b.n_packets;
    p.items = d_items;
    p.n_items = n_items;
    p.work = d_work;
    p.filter = ctx->dev.filter;
    p.n_uniq = h.n_uniq;
    p.counts_in_smem = counts_in_smem ? 1u : 0u;
    p.vtab_in_smem = vtab_in_smem ? 1u : 0u;
    p.vtab = ctx->dev.vtab;
    p.vtab_words = h.vtab_words;
    p.vt_slots_a = h.vtab[1]; p.vt_shift_a = h.vtab[2];
    p.vt_slots_b = h.vtab[3]; p.vt_shift_b = h.vtab[4];
    p.vt_one = h.vtab[5]; p.vt_rec = h.vtab[6]; p.vt_blob = h.vtab[7];
    p.mul64 = 64u;
    p.mul4096 = 4096u;
    for (int k = 0; k < 4; k++) p.sel[k] = 0x80u << (8 * k);
    p.uniq_counts = (unsigned long long *)d_uniq_counts;
    p.pat_to_uniq = ctx->dev.pat_to_uniq;
    p.n_pat = h.n_pat;
    p.n_out = out.n;
    for (int r = 0; r < KMPB_MAX_OUT; r++) p.out[r] = out.vec[r];
    const uint32_t warps_needed = n_items;
    int grid = (int)std::min<uint32_t>((uint32_t)ctx->sm_count, (warps_needed + UN_WARPS - 1) / UN_WARPS);
    if (grid < 1) grid = 1;
    if (ctx->profile) KMPB_CUDA(cudaEventRecord(ctx->ev_kernel[0], stream));
    if (find) kmpb_union_find_kernel<<<grid, UN_THREADS, smem_bytes, stream>>>(p, *find);
    else kmpb_union_kernel<<<grid, UN_THREADS, smem_bytes, stream>>>(p);
    if (ctx->profile) KMPB_CUDA(cudaEventRecord(ctx->ev_kernel[1], stream));
    ctx->launches += 2;
    KMPB_CUDA(cudaGetLastError());
    return KMPB_OK;
}
