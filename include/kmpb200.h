/*
 * kmpb200.h -- C ABI of libkmpb200.so, the B200 (sm_100a) replacement for the KMP packet-matching
 * hot path of Lemnon95/multithreading_string_matching.
 *
 * The reference has no library / plugin / FFI interface: its hot path is two file-local functions
 * (kmp_prefix, kmp_matcher) copy-pasted into five stand-alone main() programs, fed by a pattern
 * loader and a libpcap ingest loop written inline in each main().  The entry points below are the
 * batch forms of exactly those pieces; every declaration cites the reference lines it replaces
 * (paths relative to the reference checkout).  INTEGRATION.md shows the call sequence a maintainer
 * of serial.c / openmp_data.c would write against this header.
 *
 * Conventions
 *   - plain C types only: pointers and sizes, no C++/torch types;
 *   - every function returns 0 on success or a negative KMPB_E* code; kmpb_last_error() returns a
 *     thread-local message for the last failure (the reference prints and exit(1)s; the CLI in
 *     csrc/host/main.c converts codes back into the reference's messages and exit status);
 *   - the caller owns every input buffer and every output array; the library owns device memory,
 *     streams and events inside the opaque context;
 *   - one context per GPU, used from one host thread at a time (the reference's kmp_matcher is
 *     re-entrant, openmp_data.c:157-164; here parallelism lives inside the device);
 *   - there is NO CPU fallback: every matching entry point fails with KMPB_ENODEVICE when no
 *     sm_100-class CUDA device is usable.
 *
 * Semantics (bit-exact with serial.c on the same inputs; see DESIGN.md section 2)
 *   - a packet's text is payload[0 .. min(first NUL byte, payload_len))        serial.c:191
 *   - occurrences are counted with overlaps ("aa" in "aaaa" = 3)               serial.c:203-206
 *   - patterns are counted independently; duplicated patterns each get the count
 *   - bytes are compared exactly, or after ASCII case folding for a KMPB_PAT_NOCASE pattern (kmpb_set_patterns_ex)
 *   - a pattern may be restricted to start offsets [lo, hi] of each payload (kmpb_set_patterns_win)
 *   - counts are 64-bit here (C int in the reference, serial.c:103).
 */
#ifndef KMPB200_H
#define KMPB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define KMPB_VERSION "0.1.0"

/* error codes */
#define KMPB_OK 0
#define KMPB_EINVAL (-1)    /* bad argument (NULL pointer, pattern longer than 99 bytes, ...) */
#define KMPB_ENOMEM (-2)    /* host or device allocation failed */
#define KMPB_ECUDA (-3)     /* a CUDA runtime call failed; message has the CUDA error string */
#define KMPB_ENODEVICE (-4) /* no usable sm_100 device: the library never falls back to the CPU */
#define KMPB_EIO (-5)       /* cannot open / read a file (errno is preserved) */
#define KMPB_EFORMAT (-6)   /* not a classic pcap savefile, truncated record, NUL in strings file */
#define KMPB_ESTATE (-7)    /* call sequence error, e.g. count before set_patterns */
#define KMPB_ELIMIT (-8)    /* a documented limit was exceeded (see DESIGN.md section 7) */

#define KMPB_MAX_PATTERN_LEN 99 /* char str[100] + fscanf("%s"), serial.c:64-66 */
/* Every packet of a batch must be shorter than this: 2 GiB - 1 MiB.  (The union engine's work items then always span
 * less than 2^31 bytes, which its 32-bit item-relative positions need.) */
#define KMPB_PACKET_LIMIT ((1ull << 31) - (1ull << 20))

#define KMPB_PROTO_UDP 0 /* dump_UDP_packet, packet_dumping.h:87-139 (default, serial.c:31) */
#define KMPB_PROTO_TCP 1 /* dump_TCP_packet, packet_dumping.h:150-188 */

/* match engines (kmpb_set_engine) */
#define KMPB_ENGINE_AUTO 0    /* = KMPB_ENGINE_UNION */
#define KMPB_ENGINE_PERPAT 1  /* one byte-indexed KMP DFA per pattern staged in shared memory; the
                                 payload is walked once per pattern, exactly the reference's
                                 packet x pattern double loop (serial.c:153-155) */
#define KMPB_ENGINE_UNION 2   /* the per-pattern KMP automata merged into their union automaton
                                 behind a shift-and prefilter; the payload is read once */

typedef struct kmpb_ctx kmpb_ctx;

const char *kmpb_version(void);
const char *kmpb_last_error(void);
/* number of usable (compute capability 10.x) CUDA devices; 0 when there is none */
int kmpb_device_count(void);
/* CUDA ordinal of the index-th usable device (0 <= index < kmpb_device_count()), -1 beyond: what kmpb_create wants when
 * a box also holds GPUs this library has no code for.  The MPI variant's rank -> host mapping (mpi_dumping.c:29-31). */
int kmpb_device_ordinal(int index);

/* ---- context ------------------------------------------------------------------------------ */
/* Replaces nothing in the reference (it has no state); owns the device buffers, streams, tables.
 * device = CUDA ordinal.  The MPI variant's MPI_Init / rank (mpi_dumping.c:29-31) maps to one
 * context per GPU. */
int kmpb_create(kmpb_ctx **out, int device);
void kmpb_destroy(kmpb_ctx *ctx);
int kmpb_set_engine(kmpb_ctx *ctx, int engine);
int kmpb_get_device(const kmpb_ctx *ctx);

/* ---- patterns: replaces the kmp_prefix loop ----------------------------------------------- */
/* serial.c:148-152 (for each pattern: prefix_array[i] = kmp_prefix(pattern)) and the table setup of
 * every rank in mpi_dumping.c:192-195.  blob holds the n_pat patterns back to back, pattern i is
 * blob[pat_off[i] .. pat_off[i+1]); 1..99 bytes each, no NUL bytes.  The failure tables are built on
 * the device, then expanded into the transition tables of both engines.  May be called again to
 * replace the set.  n_pat == 0 is valid (every count call then returns no counts). */
int kmpb_set_patterns(kmpb_ctx *ctx, const uint8_t *blob, const uint32_t *pat_off, uint32_t n_pat);

/* Per-pattern flags (kmpb_set_patterns_ex).  KMPB_PAT_NOCASE: the pattern matches at position k of a packet's text when
 * fold(text[k+j]) == fold(p[j]) for every j, where fold maps A-Z (0x41-0x5A) to a-z and leaves every other byte as it
 * is: no other pair of bytes that differ in bit 5 folds (@ `, [ {, \ |, ] }, ^ ~, _ DEL, and every byte >= 0x80: no
 * locale, no Latin-1).  The text still ends at its first NUL, occurrences still overlap ("aA" nocase in "AaAa" = 3) and
 * lie inside one packet.  Two patterns are the same distinct pattern iff they have the same flag and are equal, after
 * folding when nocase, byte for byte when not: "Ack", "ACK" and "ack", all nocase, are one (each gets the full count,
 * their find records carry the lowest file-order index of the three); "ack" case-sensitive and "ACK" nocase are two,
 * and one text occurrence of "ack" yields a record for each.  kmpb_get_prefix of a nocase pattern returns the failure
 * table of its folded form.  Every count and find form, the savefile pipeline and kmpb_stream_* honour the flags. */
#define KMPB_PAT_NOCASE 1u
/* kmpb_set_patterns with flags[n_pat], one byte per pattern; flags == NULL is exactly kmpb_set_patterns.  A bit other
 * than KMPB_PAT_NOCASE is KMPB_EINVAL, naming the pattern. */
int kmpb_set_patterns_ex(kmpb_ctx *ctx, const uint8_t *blob, const uint32_t *pat_off, uint32_t n_pat, const uint8_t *flags);
/* Position windows (kmpb_set_patterns_win).  A pattern with window [lo, hi] matches at offset o of a packet iff it
 * matches there under the rules above (the text ends at the first NUL, occurrences overlap and lie inside one packet,
 * case folding when nocase) and lo <= o <= hi: its count is the number of its unwindowed matches whose first byte lies
 * at a payload offset in [lo, hi], its find records exactly those matches, and a packet is selected iff it holds a
 * counted match of any pattern, windowed or not.  {0, KMPB_WINDOW_ANY} is no window: the pattern behaves as in
 * kmpb_set_patterns_ex.  Otherwise 0 <= lo <= hi <= KMPB_WINDOW_MAX; anything else (lo > hi, hi above KMPB_WINDOW_MAX, a
 * window open at the top: lo > 0 with hi = KMPB_WINDOW_ANY) is KMPB_EINVAL, naming the pattern.  Two patterns are the
 * same distinct pattern iff they have the same bytes (folded when nocase), the same flag and the same window: "GET"
 * unwindowed and "GET" in [0, 0] are two, and an occurrence at offset 0 yields a record for each.  kmpb_get_prefix does
 * not depend on the window.  The union engine matches the windowed patterns in a pass of their own that reads only each
 * packet's first max(hi + pattern length) bytes; every count, find and select form and kmpb_stream_* honour the
 * windows. */
typedef struct kmpb_window {
    uint32_t lo, hi;
} kmpb_window;
#define KMPB_WINDOW_ANY 0xffffffffu
#define KMPB_WINDOW_MAX 65535u
/* kmpb_set_patterns_ex with win[n_pat], one window per pattern; win == NULL is exactly kmpb_set_patterns_ex.  Refused
 * with KMPB_ESTATE while a frame stream is open, like the other pattern calls. */
int kmpb_set_patterns_win(kmpb_ctx *ctx, const uint8_t *blob, const uint32_t *pat_off, uint32_t n_pat, const uint8_t *flags,
                          const kmpb_window *win);
uint32_t kmpb_pattern_count(const kmpb_ctx *ctx);
/* The device-built failure table of pattern i, copied back as the int[m] that kmp_prefix returns
 * (serial.c:217-238).  pi_out must hold m = pat_off[i+1]-pat_off[i] entries. */
int kmpb_get_prefix(kmpb_ctx *ctx, uint32_t pattern_index, int32_t *pi_out, uint32_t capacity);

/* ---- matching: replaces the packet x pattern loop ----------------------------------------- */
/* serial.c:153-155 / openmp_data.c:157-175 / mpi_dumping.c:198-200:
 *     for k in packets: for i in patterns: count[i] += kmp_matcher(payload[k], pattern[i], pi[i])
 * The payloads come as one flat CSR batch instead of N malloc'd buffers (serial.c:124-137):
 * packet k is bytes[offsets[k] .. offsets[k+1]), offsets has n_packets+1 non-decreasing entries, and every
 * packet is shorter than KMPB_PACKET_LIMIT.  Every host form -- kmpb_count_host, kmpb_find_host, the savefile forms
 * (a payload is its frame's captured length less the headers) and kmpb_stream_push -- checks each packet before
 * anything runs and returns KMPB_ELIMIT naming it.
 *
 * Host form: bytes / offsets are host memory (pinned memory from kmpb_host_alloc is copied
 * asynchronously in chunks on several streams, overlapped with the match kernels; pageable memory
 * works but is slower).  counts_out[n_pat] is overwritten with this batch's counts.  Synchronous. */
int kmpb_count_host(kmpb_ctx *ctx, const uint8_t *bytes, const uint64_t *offsets, uint64_t n_packets,
                    uint64_t *counts_out);

/* Device form: d_bytes (32-byte aligned, readable up to total_bytes rounded up to 32) and d_offsets
 * (values below 2^56, at most 64 GiB between the first and the last: KMPB_ELIMIT otherwise)
 * are device memory on the context's GPU; d_counts[n_pat] (device, uint64) is ACCUMULATED into, so
 * a caller can sum several batches and all-reduce once (mpi_dumping.c:202).  Asynchronous on
 * `stream` (a cudaStream_t passed as void*; NULL = CUDA's default stream, as in the runtime API).
 * Device-form calls (kmpb_count_device*, kmpb_find_device_span, kmpb_select_device_span) on one context share scratch buffers, so they run on the
 * device in call order, whatever streams they are issued on: each call's work waits, on the device, for the work of the
 * one issued before it.  The host forms and kmpb_stream_open run after every device-form call issued before them.  Work
 * of the caller's own on other streams is not ordered by this: order it with events as usual. */
int kmpb_count_device(kmpb_ctx *ctx, const uint8_t *d_bytes, const uint64_t *d_offsets,
                      uint64_t n_packets, uint64_t *d_counts, void *stream);
/* Same, for a caller that already knows first_byte = offsets[0] and end_byte = offsets[n_packets]:
 * no device-to-host read, so the call never synchronises. */
int kmpb_count_device_span(kmpb_ctx *ctx, const uint8_t *d_bytes, const uint64_t *d_offsets,
                           uint64_t n_packets, uint64_t first_byte, uint64_t end_byte,
                           uint64_t *d_counts, void *stream);
/* Same, with the reduce across GPUs inside the match kernel: the counts are added to n_vectors (1..8)
 * count vectors of uint64[n_pat] -- this GPU's own and those of its peers, mapped into this process
 * over NVLink (CUDA IPC / symmetric memory) -- by system-scope atomics issued by the kernel's last
 * block (union engine) or by the count expansion that follows the match kernel (per-pattern engine).  Replaces the local merge (openmp_data.c:169-173) plus MPI_Reduce(SUM) (mpi_dumping.c:202)
 * for device-resident callers: when every rank has passed its own batch, every vector holds the
 * total.  The caller orders "all ranks have finished" (a barrier) before reading a vector. */
int kmpb_count_device_span_peers(kmpb_ctx *ctx, const uint8_t *d_bytes, const uint64_t *d_offsets,
                                 uint64_t n_packets, uint64_t first_byte, uint64_t end_byte,
                                 uint64_t *const *d_counts_all, uint32_t n_vectors, void *stream);
/* The device forms never wait, so they cannot report what only the device knows: a packet of KMPB_PACKET_LIMIT bytes or
 * more (outside the documented limits: the union engine's counts and records of that batch are unspecified).  This call
 * waits for the context's device and returns KMPB_ELIMIT if any union-engine device-form call since the last check met
 * one; the check clears what it reports.  (The host forms check every packet before anything runs: they never set it.) */
int kmpb_check_device_errors(kmpb_ctx *ctx);
/* Device copy of the per-pattern counts of the last kmpb_count_host call (uint64[n_pat] on the
 * context's GPU), for callers that combine several GPUs with a collective (mpi_dumping.c:202). */
uint64_t *kmpb_device_counts(kmpb_ctx *ctx);

/* Profiling hooks for bench.py: with profile on, the dominant match kernel of each count call (with windowed patterns:
 * the window kernel and the union kernel together) is bracketed by CUDA events on the stream it is launched on; kmpb_last_kernel_ms waits for and returns
 * the duration of the most recent one (device-form calls only). */
int kmpb_set_profile(kmpb_ctx *ctx, int on);
int kmpb_last_kernel_ms(kmpb_ctx *ctx, double *ms_out);
/* Number of kernel launches issued by this context so far (bench.py reports it). */
uint64_t kmpb_launch_count(const kmpb_ctx *ctx);
/* Device time in milliseconds of the most recent kmpb_count_host call, measured with CUDA events on
 * the context's streams: [0] whole call (H2D + kernels + D2H), [1] match kernels only. */
int kmpb_last_timing(const kmpb_ctx *ctx, double *ms_out, int n);

/* ---- finding: where the patterns occur ----------------------------------------------------- */
/* The count entry points say how often each pattern occurs; the find entry points say where.  A match is one
 * occurrence that the count forms count, no more and no less: it lies inside one packet, no NUL byte comes before its
 * end in that packet (serial.c:191), and overlapping occurrences are separate matches.  Each match is one record:
 *   packet   index of the packet in the caller's batch (kmpb_find_pcap: among the accepted packets, the numbering of
 *            kmpb_pcap_packets and of kmpb_count_pcap's first / count);
 *   offset   byte offset of the match's first byte inside that packet's payload;
 *   pattern  the lowest file-order index among the patterns equal to the matched one (a token listed three times
 *            yields one record per occurrence, carrying the index of its first listing).
 * So for every pattern i, the count kmpb_count_host reports for i on the same batch equals the number of records whose
 * pattern is the first index of i's token.  "Sorted" means ordered by (packet, offset, pattern).
 * Finding always runs the union engine, whatever kmpb_set_engine selected (the per-pattern engine only counts).
 * n_pat == 0 or an empty batch is valid and yields 0 matches.  Errors: KMPB_ESTATE before kmpb_set_patterns,
 * KMPB_EINVAL for a NULL pointer or an unknown flag, KMPB_ENODEVICE without a B200. */
typedef struct kmpb_match {
    uint64_t packet;
    uint32_t offset;
    uint32_t pattern;
} kmpb_match; /* 16 bytes */

#define KMPB_FIND_SORTED 1u /* kmpb_find_device_span: sort the records (device radix sort, scratch owned by the context) */

/* Device form, asynchronous on `stream` like kmpb_count_device_span and with its preconditions and limits (d_bytes
 * 32-byte aligned, at most 2^31-1 packets, offsets below 2^56, at most 64 GiB in one batch).  d_out (device,
 * kmpb_match[capacity]) receives records [0, min(total, capacity)); *d_n_found (device, uint64) is OVERWRITTEN with the
 * total number of matches, which may exceed capacity.  With KMPB_FIND_SORTED and no overflow the records are sorted;
 * the sort costs time in proportion to `capacity`, so size the buffer close to the total (the sum of the kmpb_count_*
 * counts of the batch is exact).  On overflow the records written are an unspecified subset of the matches, in no
 * particular order: run again with a larger buffer.  Unsorted, the records come in an unspecified order.  It shares
 * scratch buffers with the count forms and is ordered with them like every device-form call (kmpb_count_device). */
int kmpb_find_device_span(kmpb_ctx *ctx, const uint8_t *d_bytes, const uint64_t *d_offsets, uint64_t n_packets,
                          uint64_t first_byte, uint64_t end_byte, kmpb_match *d_out, uint64_t capacity,
                          uint64_t *d_n_found, uint32_t flags, void *stream);
/* Host form: synchronous, chunked and overlapped like kmpb_count_host (KMPB_CHUNK_MB sets the chunk size), always
 * sorted.  out (host, kmpb_match[capacity]) receives the first min(total, capacity) records in sorted order and
 * *n_found the total.  The device record buffers grow as needed; a chunk whose records overflowed them is matched
 * again from the copy already on the device. */
int kmpb_find_host(kmpb_ctx *ctx, const uint8_t *bytes, const uint64_t *offsets, uint64_t n_packets,
                   kmpb_match *out, uint64_t capacity, uint64_t *n_found);

/* ---- the data-parallel split of the MPI variant -------------------------------------------- */
/* mpi_dumping.c:149-157: every rank gets n_packets / world packets, rank 0 also the remainder;
 * slices are contiguous in packet order.  Pure arithmetic, usable without a GPU. */
void kmpb_shard_range(uint64_t n_packets, uint32_t world, uint32_t rank, uint64_t *first, uint64_t *count);

/* ---- pinned host memory for the packer ------------------------------------------------------ */
void *kmpb_host_alloc(size_t bytes); /* cudaHostAlloc; NULL on failure */
void kmpb_host_free(void *p);

/* ---- host side of the path (plain C, no GPU needed) ---------------------------------------- */
/* dump_UDP_packet (packet_dumping.h:87-139) / dump_TCP_packet (:150-188) as offset + length inside
 * the frame.  Return 1 if the reference returns a payload, 0 if it returns NULL. */
int kmpb_extract_udp(const uint8_t *frame, uint32_t frame_len, uint32_t *payload_off, uint32_t *payload_len);
int kmpb_extract_tcp(const uint8_t *frame, uint32_t frame_len, uint32_t *payload_off, uint32_t *payload_len);

typedef struct kmpb_patterns {
    uint8_t *blob;     /* tokens back to back */
    uint32_t *pat_off; /* n_pat + 1 offsets */
    uint32_t n_pat;
} kmpb_patterns;
/* The fscanf("%s") token loop, serial.c:54-87: whitespace-separated tokens in file order,
 * duplicates kept.  KMPB_EIO if the file cannot be opened (errno kept for perror), KMPB_EFORMAT for
 * a token over 99 bytes or a NUL byte. */
int kmpb_load_patterns_file(const char *path, kmpb_patterns *out);
void kmpb_free_patterns(kmpb_patterns *p);

typedef struct kmpb_csr {
    uint8_t *bytes;      /* accepted payloads back to back; padded with >= 64 zero bytes */
    uint64_t *offsets;   /* n_packets + 1 */
    uint64_t n_packets;  /* frames whose payload the extractor accepted */
    uint64_t n_frames;   /* records in the savefile */
    uint64_t total_bytes;
    int pinned;          /* 1: cudaHostAlloc memory, 0: malloc */
} kmpb_csr;
/* The pcap_open_offline / pcap_next_ex ingest loop, serial.c:91-141 (openmp_data.c:94-147): reads a
 * classic pcap savefile (either byte order, usec or nsec) or a pcapng file, extracts every frame's payload with the
 * chosen extractor over its captured length and packs the accepted payloads into a flat CSR batch,
 * in pinned memory when `pinned` is non-zero.  KMPB_EIO / KMPB_EFORMAT on failure. */
int kmpb_load_pcap_csr(const char *path, int proto, int pinned, kmpb_csr *out);
void kmpb_free_csr(kmpb_csr *csr);

/* The same ingest loop fused with the match loop, serial.c:91-155 (the producer/consumer shape of
 * openmp_task.c:113-178: batches of packets are matched while the next batch is being read).
 * kmpb_pcap_open maps the savefile, frames its records and locates the accepted payloads (one
 * sequential pass, nothing copied).  kmpb_count_pcap counts the patterns in accepted packets
 * [first, first+count) -- a rank's slice as kmpb_shard_range gives it, or everything -- by packing
 * ~64 MiB batches of payloads into pinned staging buffers (all host threads), copying each to the
 * device and matching it while the next one is packed.  counts_out[n_pat] is caller-owned. */
typedef struct kmpb_pcap kmpb_pcap;
int kmpb_pcap_open(const char *path, int proto, kmpb_pcap **out);
void kmpb_pcap_close(kmpb_pcap *pc);
uint64_t kmpb_pcap_packets(const kmpb_pcap *pc); /* frames whose payload the extractor accepted */
uint64_t kmpb_pcap_frames(const kmpb_pcap *pc);  /* records in the file */
uint64_t kmpb_pcap_bytes(const kmpb_pcap *pc);   /* sum of the accepted payload lengths */
int kmpb_count_pcap(kmpb_ctx *ctx, const kmpb_pcap *pc, uint64_t first, uint64_t count, uint64_t *counts_out);
/* Optional: allocate the device and pinned host staging buffers of the chunked forms (kmpb_count_host, kmpb_count_pcap,
 * kmpb_stream_*) ahead of time, for batches of up to max_batch_bytes payload bytes and max_packets packets (0, 0: the
 * defaults of kmpb_count_pcap) -- e.g. while another thread is still reading the savefile (serial.c:91-141); pinned
 * allocations take a few hundred milliseconds.  The counting calls grow the buffers themselves when they must. */
int kmpb_reserve_staging(kmpb_ctx *ctx, uint64_t max_batch_bytes, uint64_t max_packets);
/* kmpb_find_host for accepted packets [first, first+count) of a savefile, through kmpb_count_pcap's packing pipeline:
 * always sorted, `packet` is the accepted-packet index (first + position in the slice). */
int kmpb_find_pcap(kmpb_ctx *ctx, const kmpb_pcap *pc, uint64_t first, uint64_t count, kmpb_match *out, uint64_t capacity,
                   uint64_t *n_found);
/* The capture record number (0-based, counting every record of the file, accepted or not) of accepted packets
 * [first, first+count) into frames_out[count]: the frame a match's packet came from (Wireshark numbers frames from 1).
 * Savefiles of 2^32 records or more are outside the documented limits. */
int kmpb_pcap_frame_index(const kmpb_pcap *pc, uint64_t first, uint64_t count, uint64_t *frames_out);

/* ---- selecting: which packets match -------------------------------------------------------- */
/* A packet is SELECTED iff it holds at least one match that the count forms count, under each pattern's case flag:
 * exactly the packets that kmpb_find_* on the same batch yields a record for.  Selecting always runs the union engine,
 * like finding; one pass gives the per-packet verdicts and, when asked for, the counts.  Its match kernel sets one bit
 * per match in a start-position bitmap of the batch (one bit per payload byte: span / 8 bytes of device memory, 1.75 GB
 * for a 14 GB batch, 8 GiB at the 64 GiB limit), which a verdict pass turns into one flag per packet and leaves zero
 * again.  The device form uses the bitmap of the context's first stream slot; the host and savefile forms one per stream
 * slot their chunk plan uses, as long as the largest chunk (a chunk can be a single packet of close to 2 GiB: 256 MiB).  All of it is owned
 * by the context and grows on demand.  Errors: KMPB_ESTATE before kmpb_set_patterns or while a frame stream is open,
 * KMPB_EINVAL for a NULL pointer or an unknown flag, KMPB_ENODEVICE without a B200. */
#define KMPB_SELECT_INVERT 1u /* kmpb_select_device_span: d_index lists the packets that are NOT selected */
/* Device form: asynchronous on `stream`, with the preconditions, limits and call-order rules of kmpb_count_device_span
 * (a packet of KMPB_PACKET_LIMIT bytes or more is reported by kmpb_check_device_errors).  d_flags[n_packets] (uint8,
 * device) is OVERWRITTEN: 1 = the packet is selected, 0 = not.  d_index (uint64[n_packets], device, may be NULL)
 * receives the ascending indices of the selected packets (KMPB_SELECT_INVERT: of the others), and *d_n_selected
 * (uint64, device) is overwritten with their number; d_n_selected may be NULL when d_index is (the verdicts alone).
 * d_counts may be NULL; when given, it is ACCUMULATED into exactly as kmpb_count_device_span does. */
int kmpb_select_device_span(kmpb_ctx *ctx, const uint8_t *d_bytes, const uint64_t *d_offsets, uint64_t n_packets,
                            uint64_t first_byte, uint64_t end_byte, uint8_t *d_flags, uint64_t *d_index,
                            uint64_t *d_n_selected, uint64_t *d_counts, uint32_t flags, void *stream);
/* Host form: synchronous, chunked and overlapped like kmpb_count_host (KMPB_CHUNK_MB sets the chunk size; a packet of
 * KMPB_PACKET_LIMIT bytes or more is KMPB_ELIMIT before anything runs).  flags_out[n_packets] (host) is overwritten
 * with the verdicts, *n_selected (may be NULL) with the number of selected packets; counts_out[n_pat] may be NULL, and
 * when given is overwritten with the batch's counts, as kmpb_count_host does. */
int kmpb_select_host(kmpb_ctx *ctx, const uint8_t *bytes, const uint64_t *offsets, uint64_t n_packets,
                     uint8_t *flags_out, uint64_t *n_selected, uint64_t *counts_out);
/* The same for accepted packets [first, first+count) of a savefile, through kmpb_count_pcap's packing pipeline:
 * flags_out[j] is the verdict of accepted packet first + j. */
int kmpb_select_pcap(kmpb_ctx *ctx, const kmpb_pcap *pc, uint64_t first, uint64_t count,
                     uint8_t *flags_out, uint64_t *n_selected, uint64_t *counts_out);
/* Plain C, no GPU: writes the capture records of the accepted packets [first, first+count) of `pc` for which
 * (flags[j] != 0) != (invert != 0) to out_path, as a savefile of the input's format, byte for byte as they are in the
 * input, in file order.  A classic savefile keeps its 24-byte header (byte order, usec / nsec magic, snaplen, link
 * type) and every chosen record (header and captured bytes, a record cut short by its snaplen as it is).  A pcapng file
 * keeps every block that holds no packet (section headers, interface descriptions, name resolution, statistics, ...) in
 * file order and the chosen packet blocks (enhanced, simple, obsolete packet blocks), so every section and its
 * interface numbering stay valid; a section header's Section Length is written as -1 (not specified), since the
 * section is shorter than the input's.  Frames whose payload the extractor refused are in neither output, inverted or not;
 * nor is whatever the ingest walk stops at (a truncated record, a malformed block) or follows it.  *n_written (may be
 * NULL) receives the number of records written.  KMPB_EINVAL when out_path names the input file itself (it is mapped
 * while it is read), KMPB_EIO when the file cannot be written; on failure no partial output is left behind. */
int kmpb_pcap_write_selected(const kmpb_pcap *pc, uint64_t first, uint64_t count, const uint8_t *flags, int invert,
                             const char *out_path, uint64_t *n_written);

/* Frames arriving one at a time (live_openmp_task.c:160-217: pcap_next in a loop, batches handed to
 * tasks while the capture goes on).  kmpb_stream_push runs the extractor on one captured frame and
 * appends the accepted payload to the current batch in pinned memory; a full batch (batch_bytes, 0 =
 * 8 MiB) is copied to the device and matched asynchronously while the caller keeps pushing.
 * kmpb_stream_flush submits the partial batch, waits, and returns the counts accumulated since
 * kmpb_stream_open in counts_out[n_pat]; pushing may continue afterwards.  One producer thread.
 * An open stream owns its context until kmpb_stream_close: its counts and its partly filled batch live in the context's
 * per-slot counters and pinned staging buffers, which every other matching call reuses.  So while a stream is open,
 * kmpb_set_patterns(_ex), every count, find and select form, kmpb_reserve_staging and a second kmpb_stream_open return
 * KMPB_ESTATE without touching it; kmpb_set_engine, the getters, kmpb_get_prefix, kmpb_check_device_errors and
 * kmpb_synth_fill_device still work.  Other work during a capture takes a second context.  Close every stream of a
 * context before kmpb_destroy. */
typedef struct kmpb_stream kmpb_stream;
int kmpb_stream_open(kmpb_ctx *ctx, int proto, uint64_t batch_bytes, kmpb_stream **out);
int kmpb_stream_push(kmpb_stream *st, const uint8_t *frame, uint32_t captured_len);
int kmpb_stream_flush(kmpb_stream *st, uint64_t *counts_out);
uint64_t kmpb_stream_packets(const kmpb_stream *st); /* payloads accepted so far */
void kmpb_stream_close(kmpb_stream *st);

/* The report, serial.c:163-168: header line, then "pattern: N times!" for every pattern with a
 * non-zero count, in pattern order.  Writes to `stream` (a FILE*, passed as void*). */
int kmpb_print_report(void *stream, const kmpb_patterns *pats, const uint64_t *counts);

/* ---- synthetic traffic (benchmarks and tests) ---------------------------------------------- */
/* Counter-based generator of the BASELINE workloads: packet p of the stream is a function of
 * (seed, p) only, so any slice can be produced on the host or directly in device memory with the
 * same bits.  Payload bytes are printable ASCII, the last byte of every payload is 0x00, and
 * `plants` patterns (taken round-robin from the plant set) overwrite pseudo-random positions.
 * len_mode 0: every payload has payload_len bytes; 1: lengths drawn from {64:40%, 576:20%,
 * 1400:30%, 9000:10%} (BASELINE config 5).  Offsets are relative to the slice start. */
typedef struct kmpb_synth {
    uint64_t seed;
    uint32_t payload_len;
    uint32_t len_mode;
    uint32_t plants;
    const uint8_t *plant_blob;     /* may be NULL when plants == 0 */
    const uint32_t *plant_off;
    uint32_t n_plant;
} kmpb_synth;
/* bytes needed for packets [first, first+count) */
uint64_t kmpb_synth_bytes(const kmpb_synth *cfg, uint64_t first, uint64_t count);
int kmpb_synth_fill_host(const kmpb_synth *cfg, uint64_t first, uint64_t count, uint8_t *bytes, uint64_t *offsets);
/* device buffers on the context's GPU; asynchronous on the context's stream, then synchronised */
int kmpb_synth_fill_device(kmpb_ctx *ctx, const kmpb_synth *cfg, uint64_t first, uint64_t count,
                           uint8_t *d_bytes, uint64_t *d_offsets);

#ifdef __cplusplus
}
#endif
#endif
