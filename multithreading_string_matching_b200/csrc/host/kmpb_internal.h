/* kmpb_internal.h -- declarations shared by the host (C) and device (CUDA) halves of libkmpb200. */
#ifndef KMPB_INTERNAL_H
#define KMPB_INTERNAL_H

#include "kmpb200.h"

#ifdef __cplusplus
extern "C" {
#endif

/* errors.c: printf-style setter for the thread-local message behind kmpb_last_error(); returns code */
int kmpb_fail(int code, const char *fmt, ...) __attribute__((format(printf, 2, 3)));

/* ------------------------------------------------------------------------------------------------
 * automaton.c: everything the device needs to match a pattern set, built once per set on the host.
 *
 * Union automaton = the per-pattern KMP automata (serial.c:190-238) merged into one DFA over the
 * trie of all pattern prefixes (for a single pattern it IS that pattern's KMP DFA).  Duplicate
 * patterns share one "unique" id; counts are expanded back to file order at the end.
 * ---------------------------------------------------------------------------------------------- */
typedef struct kmpb_tables {
    /* patterns */
    uint32_t n_pat;          /* patterns in file order (duplicates included) */
    uint32_t n_uniq;         /* distinct patterns */
    uint32_t *pat_to_uniq;   /* [n_pat] */
    uint32_t *uniq_len;      /* [n_uniq] */
    uint32_t *uniq_off;      /* [n_uniq+1] into uniq_blob */
    uint8_t *uniq_blob;      /* a nocase pattern's bytes are folded (A-Z to a-z) */
    uint8_t *uniq_flags;     /* [n_uniq] KMPB_PAT_NOCASE or 0: part of a distinct pattern's identity */
    uint32_t n_nocase;       /* distinct nocase patterns without a window (non-zero: the union engine runs its nocase kernels) */
    uint32_t max_len, min_len;
    /* Distinct ids [0, n_union) are the patterns without a window, in the order a set without windows gives them; the
     * filter, the probe tables (vtab), the gate and the automaton below hold these alone.  Ids [n_union, n_uniq) are
     * the windowed ones (kmpb_tables_build_win), matched by the window kernel through wvtab. */
    uint32_t n_union;
    uint32_t *uniq_lo, *uniq_hi; /* [n_uniq - n_union] window of distinct id n_union + w */
    uint32_t win_lo_min, win_hi_max, win_reach; /* min lo, max hi, max(hi + len) over the windowed patterns */
    uint32_t win_nocase;     /* windowed distinct nocase patterns (wvtab then has the nocase layout) */
    uint32_t win_first[8];   /* bit c: some windowed pattern can start with byte c */
    uint32_t *wvtab;         /* the windowed patterns' probe tables, in vtab's layout (distinct ids as above) */
    uint32_t wvtab_words;

    /* byte classes: bytes that occur in no pattern share class 0 */
    uint32_t n_class;
    uint8_t byte_class[256];

    /* union DFA: next[state * n_class + class] = target state, bit 31 set when the target state
     * reports at least one pattern.  It reads the text as it is; a nocase pattern's upper-case letters go where its
     * lower-case ones go.  A set of both kinds gets the product of the two kinds' automata, and no bare trie. */
    uint32_t n_state;
    uint32_t *next;          /* [n_state * n_class] */
    /* the same states as a bare trie: trie[state * n_class + class] = child (0 = none), bit 31 set when
     * a pattern ends at the child; state_term[state] = that pattern's distinct id, or ~0 */
    uint32_t *trie;          /* [n_state * n_class] */
    uint32_t *state_term;    /* [n_state] */
    /* outputs of state s: uniq ids out_id[out_head[s] .. out_head[s+1]), longest pattern first */
    uint32_t *out_head;      /* [n_state+1] */
    uint32_t *out_id;

    /* shift-and prefilter (automaton.c kmpb_filter6_build): for byte value c, filter6[c] has bit (6*d + b) set when some
     * pattern of bucket b (0..4) has byte c at depth d (0..3) or is shorter than d+1 bytes; bit 5 of depth 0 is set for
     * c == 0 only and bit 5 of depths 1..3 always (the NUL detector); bits 24..29 always (a report lingers one step, so
     * that the kernel can update its state once per two bytes) */
    uint32_t filter6[256];
    double filter6_fp_estimate;    /* estimated candidate probability per text byte, uniform bytes */

    /* start-anchored verification tables (the device's slow path): two probe tables -- A for the two-byte patterns,
     * keyed by their two bytes, B for the patterns of three and more bytes, keyed by their first three -- of slots
     * {first record, records}; a text position probes one slot of each and compares the records of those slots.
     * Layout of vtab (u32 words):
     *   [0] total words
     *   [1] word offset of the slots of A (0 = no two-byte patterns)   [2] hash shift of A (slots = 1 << (32 - shift))
     *   [3] word offset of the slots of B (0 = none)                   [4] hash shift of B
     *   [5] word offset of the one-byte patterns' table (256 words: distinct id or 0xffffffff, by text byte), 0 = there
     *       are none; in a set with a nocase pattern 512 words, the second 256 for the nocase one-byte patterns
     *   [6] word offset of the records   [7] word offset of the pattern words
     *   records (8 words, 16-byte aligned): {pattern bytes 0..3, mask of those that exist, bytes 4..7, their mask,
     *            length, distinct id, word offset of the pattern's bytes inside the pattern words, tail masks}
     *   pattern words: every pattern zero-padded to a multiple of 4 bytes
     *   tail masks: for a nocase pattern of more than 8 bytes, one mask word per pattern word (0xdf at its letters, 0xff
     *            at its other bytes, 0 past its end); the record's last word is their vtab word offset, else 0.
     * A nocase pattern is stored folded, its masks clear bit 5 at its letters, and it has a record in the slot of every
     * case variant of its key (up to 4 in A, 8 in B; once per distinct slot). */
    uint32_t *vtab;
    uint32_t vtab_words;

    /* prefix gate (automaton.c build_gate): a hashed bitmap that every position at which some pattern starts passes.
     * Word kmpb_gate_slot(first two bytes, gate_shift) of a position; in it, a pattern of three and more bytes sets bit
     * 31 - (third byte & 31), a two-byte pattern every bit, a one-byte pattern every bit of the words of all 256 second
     * bytes; a nocase pattern does so for every case variant of its first two bytes.  gate_words = 0: no gate (too full to be worth its lookups: the resolve step re-runs the filter instead). */
    uint32_t *gate;
    uint32_t gate_words, gate_shift;
} kmpb_tables;

/* pcap_csr.c, used by the streamed savefile path (api.cu): end of the chunk of whole packets that starts at
 * `first`, holds at most max_bytes payload bytes (at least one packet) and max_packets packets and stops
 * before `last`; packs packets [first, first+count) back to back into dst, offsets[0..count] from 0 */
uint64_t kmpb_pcap_chunk_end(const kmpb_pcap *pc, uint64_t first, uint64_t last, uint64_t max_bytes, uint64_t max_packets,
                             uint64_t *bytes_out);
void kmpb_pcap_pack(const kmpb_pcap *pc, uint64_t first, uint64_t count, uint8_t *dst, uint64_t *offsets);
/* the first accepted packet in [first, first+count) whose payload is min_len bytes or longer, else first+count (a
 * payload is its frame's captured length less the headers: a savefile can hold one of any size up to 4 GiB) */
uint64_t kmpb_pcap_first_long(const kmpb_pcap *pc, uint64_t first, uint64_t count, uint64_t min_len);

/* slot of a key (a text position's first two or three bytes) in a probe table (the device uses the same expression) */
uint32_t kmpb_vtab_slot(uint32_t key, uint32_t shift);
/* word of the prefix gate for a text position whose first bytes are the low bytes of x (only the low two matter: the
 * multiplier's low 16 bits are zero, so the device hashes a whole text word without masking it) */
#define KMPB_GATE_MUL 0x79b10000u
uint32_t kmpb_gate_slot(uint32_t x, uint32_t shift);
int kmpb_tables_build(kmpb_tables *t, const uint8_t *blob, const uint32_t *pat_off, uint32_t n_pat);
/* ... and, with_dfa != 0, the merged automaton of all patterns the table tests compare against (never uploaded) */
int kmpb_tables_build_ex(kmpb_tables *t, const uint8_t *blob, const uint32_t *pat_off, uint32_t n_pat, int with_dfa);
/* ... with per-pattern KMPB_PAT_* flags[n_pat] (NULL = all zero, which builds word for word what kmpb_tables_build does) */
int kmpb_tables_build_flags(kmpb_tables *t, const uint8_t *blob, const uint32_t *pat_off, uint32_t n_pat,
                            const uint8_t *flags, int with_dfa);
/* ... with per-pattern windows win[n_pat] (NULL = none, which builds word for word what kmpb_tables_build_flags does) */
int kmpb_tables_build_win(kmpb_tables *t, const uint8_t *blob, const uint32_t *pat_off, uint32_t n_pat,
                          const uint8_t *flags, const kmpb_window *win, int with_dfa);
/* the prefilter words (5 pattern buckets + NUL in 6-bit fields, depth 4 + a lingering field): automaton.c */
int kmpb_filter6_build(const kmpb_tables *t, uint32_t words[256], double *estimate);
void kmpb_tables_free(kmpb_tables *t);

#ifdef __cplusplus
}
#endif
#endif
