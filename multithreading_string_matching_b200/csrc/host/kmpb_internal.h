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
    uint8_t *uniq_blob;
    uint32_t max_len, min_len;

    /* byte classes: bytes that occur in no pattern share class 0 */
    uint32_t n_class;
    uint8_t byte_class[256];

    /* union DFA: next[state * n_class + class] = target state, bit 31 set when the target state
     * reports at least one pattern */
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
     *   [5] word offset of the one-byte patterns' table (256 words: distinct id or 0xffffffff), 0 = there are none
     *   [6] word offset of the records   [7] word offset of the pattern words
     *   records (8 words, 16-byte aligned): {pattern bytes 0..3, mask of those that exist, bytes 4..7, their mask,
     *            length, distinct id, word offset of the pattern's bytes inside the pattern words, 0}
     *   pattern words: every pattern zero-padded to a multiple of 4 bytes */
    uint32_t *vtab;
    uint32_t vtab_words;
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
int kmpb_tables_build(kmpb_tables *t, const uint8_t *blob, const uint32_t *pat_off, uint32_t n_pat);
/* ... and, with_dfa != 0, the merged automaton of all patterns the table tests compare against (never uploaded) */
int kmpb_tables_build_ex(kmpb_tables *t, const uint8_t *blob, const uint32_t *pat_off, uint32_t n_pat, int with_dfa);
/* the prefilter words (5 pattern buckets + NUL in 6-bit fields, depth 4 + a lingering field): automaton.c */
int kmpb_filter6_build(const kmpb_tables *t, uint32_t words[256], double *estimate);
void kmpb_tables_free(kmpb_tables *t);

#ifdef __cplusplus
}
#endif
#endif
