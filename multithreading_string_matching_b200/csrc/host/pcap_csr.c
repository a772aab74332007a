/* pcap_csr.c -- savefile ingest: the step before the hot path (serial.c:91-141, openmp_data.c:94-147).
 *
 * The reference lets libpcap frame the records (pcap_open_offline serial.c:91, pcap_next_ex :115),
 * copies every frame, extracts its payload and stores one malloc'd buffer per payload.  Here the
 * savefile is mapped (its pages faulted in by all host threads), the records are framed and their payloads
 * located in one sequential pass, and
 * the accepted payloads are then packed back to back by all host threads (OpenMP, like the
 * reference's own extraction loop at openmp_data.c:128-147) into ONE flat buffer plus an offsets
 * array -- the CSR batch the device consumes -- in pinned memory so the H2D copies can run
 * asynchronously.
 *
 * Classic savefiles (either byte order, microsecond or nanosecond stamps) and pcapng files are read.
 * Frames are read with their captured length (openmp_data.c:114-116; serial.c:117-120 uses the wire
 * length, the same number whenever caplen == len).  Like the reference's `while (pcap_next_ex(...)
 * >= 0)` loop, a truncated trailing record ends the walk without an error.
 */
#include <errno.h>
#include <fcntl.h>
#include <omp.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>

#include "kmpb_internal.h"

#define PCAP_GLOBAL_HDR 24u
#define PCAP_RECORD_HDR 16u
#define CSR_TAIL_PAD 64u

typedef int (*extract_fn)(const uint8_t *, uint32_t, uint32_t *, uint32_t *);

static uint32_t load32(const uint8_t *p, int swapped)
{
    uint32_t v;
    memcpy(&v, p, sizeof v);
    return swapped ? __builtin_bswap32(v) : v;
}

/* Where an accepted payload lies in the mapped file. */
typedef struct {
    uint64_t at;  /* file offset of the payload's first byte */
    uint32_t len;
    uint32_t frame; /* its capture record number, from 0 (a savefile of 2^32 records or more is outside the limits) */
} payload_ref;

/* Growing list of accepted payloads. */
typedef struct {
    payload_ref *refs;
    size_t cap;
    uint64_t packets, frames, bytes;
} ref_list;

/* one frame of `caplen` captured bytes at file offset `at`: run the extractor, remember the payload */
static int take_frame(ref_list *l, const uint8_t *file, size_t at, uint32_t caplen, extract_fn extract)
{
    uint32_t off, len;
    const uint64_t frame = l->frames++;
    if (!extract(file + at, caplen, &off, &len)) return KMPB_OK;
    if (l->packets == l->cap) {
        size_t cap = l->cap ? 2 * l->cap : (size_t)1 << 16;
        payload_ref *grown = realloc(l->refs, cap * sizeof *grown);
        if (!grown) return KMPB_ENOMEM;
        l->refs = grown;
        l->cap = cap;
    }
    l->refs[l->packets].at = at + off;
    l->refs[l->packets].len = len;
    l->refs[l->packets].frame = (uint32_t)frame;
    l->bytes += len;
    l->packets++;
    return KMPB_OK;
}

/* Pass 1 for a classic savefile, sequential (record n+1 starts where record n's header says): frame the
 * records, run the extractor on every frame and remember where the accepted payloads are. */
static int index_classic(const uint8_t *file, size_t size, int swapped, extract_fn extract, ref_list *l)
{
    size_t at = PCAP_GLOBAL_HDR;
    while (size - at >= PCAP_RECORD_HDR) {
        uint32_t caplen = load32(file + at + 8, swapped);
        at += PCAP_RECORD_HDR;
        if (caplen > size - at) break; /* truncated record: libpcap reports an error, the loop ends */
        /* The walk is a chain of dependent cache misses (a record header and the few header bytes the extractor reads,
         * every caplen + 16 bytes).  A guess breaks the chain: records tend to come in runs of one size, so the header
         * of the record 8 further on is probably 8 x this record's stride away -- a wrong guess costs one useless
         * prefetch. */
        {
            const size_t ahead = at + 8 * ((size_t)caplen + PCAP_RECORD_HDR);
            if (ahead < size) {
                __builtin_prefetch(file + ahead - PCAP_RECORD_HDR);
                __builtin_prefetch(file + ahead + 48);
            }
        }
        if (take_frame(l, file, at, caplen, extract) != KMPB_OK) return KMPB_ENOMEM;
        at += caplen;
    }
    return KMPB_OK;
}

/* Pass 1 for a pcapng file (what libpcap's pcap_next_ex hands out when pcap_open_offline meets one, SURVEY
 * 8f-3): blocks of [type, total length, body, total length], 32-bit aligned; a Section Header Block sets
 * the byte order of its section; packets come from Enhanced (6), Simple (3) and obsolete Packet (2)
 * blocks; everything else (interface descriptions, name resolution, statistics, ...) is skipped.  A
 * malformed or truncated block ends the walk, like a truncated record does. */
#define NG_SHB 0x0a0d0d0au
#define NG_BYTE_ORDER 0x1a2b3c4du
static int index_pcapng(const uint8_t *file, size_t size, extract_fn extract, ref_list *l)
{
    size_t at = 0;
    int swapped = 0;
    uint32_t snaplen0 = 0; /* snaplen of interface 0, for Simple Packet Blocks */
    int have_if0 = 0;
    while (size - at >= 12) {
        uint32_t type_raw;
        memcpy(&type_raw, file + at, 4);
        if (type_raw == NG_SHB) { /* palindromic: readable before the byte order is known */
            if (size - at < 28) break;
            uint32_t bom;
            memcpy(&bom, file + at + 8, 4);
            if (bom == NG_BYTE_ORDER) swapped = 0;
            else if (__builtin_bswap32(bom) == NG_BYTE_ORDER) swapped = 1;
            else break;
            have_if0 = 0;
        }
        const uint32_t type = type_raw == NG_SHB ? NG_SHB : load32(file + at, swapped);
        const uint32_t total = load32(file + at + 4, swapped);
        if (total < 12 || (total & 3u) || total > size - at) break;
        const size_t body = at + 8, body_len = total - 12;
        if (type == 1u) { /* Interface Description Block: linktype u16, reserved u16, snaplen u32 */
            if (body_len >= 8 && !have_if0) {
                snaplen0 = load32(file + body + 4, swapped);
                have_if0 = 1;
            }
        } else if (type == 6u) { /* Enhanced Packet Block: interface, ts hi, ts lo, caplen, origlen, data */
            if (body_len < 20) break;
            const uint32_t caplen = load32(file + body + 12, swapped);
            if (caplen > body_len - 20) break;
            if (take_frame(l, file, body + 20, caplen, extract) != KMPB_OK) return KMPB_ENOMEM;
        } else if (type == 2u) { /* obsolete Packet Block: interface u16, drops u16, ts hi, ts lo, caplen, len, data */
            if (body_len < 20) break;
            const uint32_t caplen = load32(file + body + 12, swapped);
            if (caplen > body_len - 20) break;
            if (take_frame(l, file, body + 20, caplen, extract) != KMPB_OK) return KMPB_ENOMEM;
        } else if (type == 3u) { /* Simple Packet Block: origlen, data (captured = min(origlen, snaplen)) */
            if (body_len < 4) break;
            uint32_t caplen = load32(file + body, swapped);
            if (have_if0 && snaplen0 && caplen > snaplen0) caplen = snaplen0;
            if (caplen > body_len - 4) caplen = (uint32_t)(body_len - 4);
            if (take_frame(l, file, body + 4, caplen, extract) != KMPB_OK) return KMPB_ENOMEM;
        }
        at += total;
    }
    return KMPB_OK;
}

/* Pass 2, parallel: offsets by a two-level prefix sum, payloads copied by all host threads (the copy
 * is what the reference does per packet at serial.c:124-137, here into one flat buffer). */
static void pack_payloads(const uint8_t *file, const payload_ref *refs, uint64_t n, uint8_t *dst, uint64_t *offsets)
{
    enum { BLOCK = 4096 };
    const uint64_t n_blocks = (n + BLOCK - 1) / BLOCK;
    uint64_t *block_base = malloc((size_t)(n_blocks + 1) * sizeof *block_base);
    if (block_base == NULL) { /* no scratch: plain sequential pack */
        uint64_t bytes = 0;
        for (uint64_t k = 0; k < n; k++) {
            offsets[k] = bytes;
            memcpy(dst + bytes, file + refs[k].at, refs[k].len);
            bytes += refs[k].len;
        }
        offsets[n] = bytes;
        return;
    }
#pragma omp parallel for schedule(static)
    for (uint64_t b = 0; b < n_blocks; b++) {
        uint64_t sum = 0, hi = (b + 1) * BLOCK < n ? (b + 1) * BLOCK : n;
        for (uint64_t k = b * BLOCK; k < hi; k++) sum += refs[k].len;
        block_base[b + 1] = sum;
    }
    block_base[0] = 0;
    for (uint64_t b = 0; b < n_blocks; b++) block_base[b + 1] += block_base[b];
#pragma omp parallel for schedule(dynamic, 4)
    for (uint64_t b = 0; b < n_blocks; b++) {
        uint64_t bytes = block_base[b], hi = (b + 1) * BLOCK < n ? (b + 1) * BLOCK : n;
        for (uint64_t k = b * BLOCK; k < hi; k++) {
            offsets[k] = bytes;
            memcpy(dst + bytes, file + refs[k].at, refs[k].len);
            bytes += refs[k].len;
        }
    }
    offsets[n] = block_base[n_blocks];
    free(block_base);
}

struct kmpb_pcap {
    const uint8_t *file;
    size_t size;
    payload_ref *refs;
    uint64_t n_packets, n_frames, total_bytes;
    dev_t dev; /* the mapped file, which kmpb_pcap_write_selected must not overwrite */
    ino_t ino;
};

int kmpb_pcap_open(const char *path, int proto, kmpb_pcap **out)
{
    if (path == NULL || out == NULL) return kmpb_fail(KMPB_EINVAL, "kmpb_pcap_open: NULL argument");
    *out = NULL;
    if (proto != KMPB_PROTO_UDP && proto != KMPB_PROTO_TCP) return kmpb_fail(KMPB_EINVAL, "unknown protocol %d", proto);
    int fd = open(path, O_RDONLY);
    struct stat st;
    if (fd < 0 || fstat(fd, &st) != 0) {
        int e = errno;
        if (fd >= 0) close(fd);
        kmpb_fail(KMPB_EIO, "%s: %s", path, strerror(e));
        errno = e;
        return KMPB_EIO;
    }
    size_t size = (size_t)st.st_size;
    if (size < PCAP_GLOBAL_HDR) {
        close(fd);
        return kmpb_fail(KMPB_EFORMAT, "truncated dump file; tried to read %u file header bytes, only got %zu",
                         PCAP_GLOBAL_HDR, size);
    }
    const uint8_t *file = mmap(NULL, size, PROT_READ, MAP_PRIVATE, fd, 0);
    close(fd);
    if (file == MAP_FAILED) return kmpb_fail(KMPB_EIO, "%s: mmap: %s", path, strerror(errno));
    madvise((void *)file, size, MADV_WILLNEED);
    /* The framing pass below is sequential (record n+1 starts where record n's header says) and touches every page of
     * the mapping once; what it would spend is mostly the page faults (10 GB in tmpfs: 0.8 s of its 0.85 s).  Faults
     * scale with threads, the walk does not: all host threads touch the pages first. */
    const int stats = getenv("KMPB_STATS") != NULL;
    const double t_map = stats ? omp_get_wtime() : 0.0;
    if (size >= ((size_t)64 << 20)) {
        const size_t page = 4096, n_pages = (size + page - 1) / page;
        unsigned long touched = 0;
#pragma omp parallel for schedule(static) reduction(+ : touched)
        for (size_t i = 0; i < n_pages; i++) touched += ((const volatile uint8_t *)file)[i * page];
        (void)touched;
    }

    uint32_t magic;
    memcpy(&magic, file, 4);
    int swapped = 0, ng = 0;
    if (magic == 0xa1b2c3d4u || magic == 0xa1b23c4du) swapped = 0;        /* usec / nsec, host order */
    else if (magic == 0xd4c3b2a1u || magic == 0x4d3cb2a1u) swapped = 1;   /* written on the other endianness */
    else if (magic == NG_SHB) ng = 1;                                     /* pcapng */
    else {
        munmap((void *)file, size);
        return kmpb_fail(KMPB_EFORMAT, "unknown file format");
    }
    extract_fn extract = proto == KMPB_PROTO_TCP ? kmpb_extract_tcp : kmpb_extract_udp;
    const double t_walk = stats ? omp_get_wtime() : 0.0;
    kmpb_pcap *pc = calloc(1, sizeof *pc);
    ref_list list = {NULL, 0, 0, 0, 0};
    if (pc == NULL || (ng ? index_pcapng(file, size, extract, &list) : index_classic(file, size, swapped, extract, &list)) != KMPB_OK) {
        free(pc);
        free(list.refs);
        munmap((void *)file, size);
        return kmpb_fail(KMPB_ENOMEM, "out of memory indexing %s", path);
    }
    pc->refs = list.refs;
    pc->n_packets = list.packets;
    pc->n_frames = list.frames;
    pc->total_bytes = list.bytes;
    pc->file = file;
    pc->size = size;
    pc->dev = st.st_dev;
    pc->ino = st.st_ino;
    *out = pc;
    if (stats)
        fprintf(stderr, "kmpb_pcap_open: %zu bytes mapped and faulted in %.3f s, %llu records framed in %.3f s\n", size,
                t_walk - t_map, (unsigned long long)list.frames, omp_get_wtime() - t_walk);
    return KMPB_OK;
}

void kmpb_pcap_close(kmpb_pcap *pc)
{
    if (pc == NULL) return;
    free(pc->refs);
    if (pc->file) munmap((void *)pc->file, pc->size);
    free(pc);
}

uint64_t kmpb_pcap_packets(const kmpb_pcap *pc) { return pc ? pc->n_packets : 0; }
uint64_t kmpb_pcap_frames(const kmpb_pcap *pc) { return pc ? pc->n_frames : 0; }
uint64_t kmpb_pcap_bytes(const kmpb_pcap *pc) { return pc ? pc->total_bytes : 0; }

int kmpb_pcap_frame_index(const kmpb_pcap *pc, uint64_t first, uint64_t count, uint64_t *frames_out)
{
    if (pc == NULL || (frames_out == NULL && count)) return kmpb_fail(KMPB_EINVAL, "kmpb_pcap_frame_index: NULL argument");
    if (first > pc->n_packets || count > pc->n_packets - first) return kmpb_fail(KMPB_EINVAL, "packet range outside the file");
    for (uint64_t k = 0; k < count; k++) frames_out[k] = pc->refs[first + k].frame;
    return KMPB_OK;
}

uint64_t kmpb_pcap_chunk_end(const kmpb_pcap *pc, uint64_t first, uint64_t last, uint64_t max_bytes, uint64_t max_packets,
                             uint64_t *bytes_out)
{
    uint64_t k = first, bytes = 0;
    while (k < last && k - first < max_packets && (k == first || bytes + pc->refs[k].len <= max_bytes)) bytes += pc->refs[k++].len;
    if (bytes_out) *bytes_out = bytes;
    return k;
}

uint64_t kmpb_pcap_first_long(const kmpb_pcap *pc, uint64_t first, uint64_t count, uint64_t min_len)
{
    for (uint64_t k = first; k < first + count; k++)
        if (pc->refs[k].len >= min_len) return k;
    return first + count;
}

void kmpb_pcap_pack(const kmpb_pcap *pc, uint64_t first, uint64_t count, uint8_t *dst, uint64_t *offsets)
{
    pack_payloads(pc->file, pc->refs + first, count, dst, offsets);
}

int kmpb_load_pcap_csr(const char *path, int proto, int pinned, kmpb_csr *out)
{
    if (path == NULL || out == NULL) return kmpb_fail(KMPB_EINVAL, "kmpb_load_pcap_csr: NULL argument");
    memset(out, 0, sizeof *out);
    kmpb_pcap *pc = NULL;
    int rc = kmpb_pcap_open(path, proto, &pc);
    if (rc != KMPB_OK) return rc;
    const uint64_t n = pc->n_packets, total = pc->total_bytes;
    size_t bytes_sz = (size_t)total + CSR_TAIL_PAD, off_sz = (size_t)(n + 1) * sizeof(uint64_t);
    uint8_t *bytes = pinned ? kmpb_host_alloc(bytes_sz) : malloc(bytes_sz);
    uint64_t *offsets = pinned ? kmpb_host_alloc(off_sz) : malloc(off_sz);
    if (bytes == NULL || offsets == NULL) {
        if (pinned) { kmpb_host_free(bytes); kmpb_host_free(offsets); }
        else { free(bytes); free(offsets); }
        kmpb_pcap_close(pc);
        return kmpb_fail(KMPB_ENOMEM, "cannot allocate %zu bytes of %s memory for the payload batch",
                         bytes_sz + off_sz, pinned ? "pinned" : "host");
    }
    pack_payloads(pc->file, pc->refs, n, bytes, offsets);
    memset(bytes + total, 0, CSR_TAIL_PAD);
    out->bytes = bytes;
    out->offsets = offsets;
    out->n_packets = n;
    out->n_frames = pc->n_frames;
    out->total_bytes = total;
    out->pinned = pinned ? 1 : 0;
    kmpb_pcap_close(pc);
    return KMPB_OK;
}

void kmpb_free_csr(kmpb_csr *csr)
{
    if (csr == NULL) return;
    if (csr->pinned) { kmpb_host_free(csr->bytes); kmpb_host_free(csr->offsets); }
    else { free(csr->bytes); free(csr->offsets); }
    memset(csr, 0, sizeof *csr);
}

/* ---- kmpb_pcap_write_selected: the chosen records, verbatim ------------------------------------------------------ */
/* The writer walks the framing once more (the ingest walk keeps no record bounds; it should not slow down for a writer
 * few callers use) with the same rules as index_classic / index_pcapng, so its n-th packet record is frame n.  Runs
 * of consecutive records to keep are written with one fwrite each. */
typedef struct {
    FILE *f;
    const uint8_t *file;
    size_t run_at, run_len; /* the pending run of bytes to write */
    int err;
    /* the chosen frames, in ascending order: frame of accepted packet first + j for the j whose verdict is chosen */
    const payload_ref *refs;
    const uint8_t *flags;
    uint64_t count, j;
    int invert;
    uint64_t next; /* the next chosen frame, UINT64_MAX when there is none */
    uint64_t frame, written;
} sel_writer;

static void next_chosen(sel_writer *w)
{
    while (w->j < w->count && (w->flags[w->j] != 0) == (w->invert != 0)) w->j++;
    w->next = w->j < w->count ? w->refs[w->j].frame : UINT64_MAX;
    w->j++;
}

static void keep(sel_writer *w, size_t at, size_t len)
{
    if (w->run_len && w->run_at + w->run_len == at) {
        w->run_len += len;
        return;
    }
    if (w->run_len && fwrite(w->file + w->run_at, 1, w->run_len, w->f) != w->run_len) w->err = 1;
    w->run_at = at;
    w->run_len = len;
}

/* bytes that are not in the input as they are: after the pending run */
static void emit(sel_writer *w, const void *bytes, size_t len)
{
    keep(w, 0, 0); /* writes the pending run, leaves none */
    if (fwrite(bytes, 1, len, w->f) != len) w->err = 1;
}

/* a Section Header Block at [at, at + total), total >= 24: copied with its Section Length set to -1 ("not specified";
 * all ones in either byte order), since the written section holds fewer blocks than the input's did */
static void section_header(sel_writer *w, size_t at, size_t total)
{
    static const uint8_t unspecified[8] = {0xff, 0xff, 0xff, 0xff, 0xff, 0xff, 0xff, 0xff};
    keep(w, at, 16);
    emit(w, unspecified, sizeof unspecified);
    keep(w, at + 24, total - 24);
}

/* a packet record at [at, at + len): the next frame */
static void packet_record(sel_writer *w, size_t at, size_t len)
{
    if (w->frame++ != w->next) return;
    keep(w, at, len);
    w->written++;
    next_chosen(w);
}

static void write_classic(sel_writer *w, size_t size, int swapped)
{
    const uint8_t *file = w->file;
    keep(w, 0, PCAP_GLOBAL_HDR);
    size_t at = PCAP_GLOBAL_HDR;
    while (size - at >= PCAP_RECORD_HDR && w->next != UINT64_MAX) {
        const uint32_t caplen = load32(file + at + 8, swapped);
        if (caplen > size - at - PCAP_RECORD_HDR) break;
        packet_record(w, at, PCAP_RECORD_HDR + (size_t)caplen);
        at += PCAP_RECORD_HDR + (size_t)caplen;
    }
}

static void write_pcapng(sel_writer *w, size_t size)
{
    const uint8_t *file = w->file;
    size_t at = 0;
    int swapped = 0;
    while (size - at >= 12) {
        uint32_t type_raw;
        memcpy(&type_raw, file + at, 4);
        if (type_raw == NG_SHB) {
            if (size - at < 28) break;
            uint32_t bom;
            memcpy(&bom, file + at + 8, 4);
            if (bom == NG_BYTE_ORDER) swapped = 0;
            else if (__builtin_bswap32(bom) == NG_BYTE_ORDER) swapped = 1;
            else break;
        }
        const uint32_t type = type_raw == NG_SHB ? NG_SHB : load32(file + at, swapped);
        const uint32_t total = load32(file + at + 4, swapped);
        if (total < 12 || (total & 3u) || total > size - at) break;
        const size_t body = at + 8, body_len = total - 12;
        if (type == 6u || type == 2u) { /* enhanced / obsolete packet block: the walk stops where index_pcapng does */
            if (body_len < 20 || load32(file + body + 12, swapped) > body_len - 20) break;
            packet_record(w, at, total);
        } else if (type == 3u) {
            if (body_len < 4) break;
            packet_record(w, at, total);
        } else if (type == NG_SHB && total >= 24) {
            section_header(w, at, total);
        } else {
            keep(w, at, total);
        }
        at += total;
    }
}

int kmpb_pcap_write_selected(const kmpb_pcap *pc, uint64_t first, uint64_t count, const uint8_t *flags, int invert,
                             const char *out_path, uint64_t *n_written)
{
    if (pc == NULL || out_path == NULL || (flags == NULL && count)) return kmpb_fail(KMPB_EINVAL, "kmpb_pcap_write_selected: NULL argument");
    if (first > pc->n_packets || count > pc->n_packets - first) return kmpb_fail(KMPB_EINVAL, "packet range outside the file");
    if (n_written) *n_written = 0;
    struct stat st;
    if (stat(out_path, &st) == 0 && st.st_dev == pc->dev && st.st_ino == pc->ino)
        return kmpb_fail(KMPB_EINVAL, "%s is the input savefile itself", out_path);
    FILE *f = fopen(out_path, "wb");
    if (f == NULL) {
        const int e = errno;
        kmpb_fail(KMPB_EIO, "%s: %s", out_path, strerror(e));
        errno = e;
        return KMPB_EIO;
    }
    setvbuf(f, NULL, _IOFBF, 1 << 20);
    sel_writer w = {f, pc->file, 0, 0, 0, pc->refs + first, flags, count, 0, invert, 0, 0, 0};
    next_chosen(&w);
    uint32_t magic;
    memcpy(&magic, pc->file, 4);
    if (magic == NG_SHB) write_pcapng(&w, pc->size);
    else write_classic(&w, pc->size, magic == 0xd4c3b2a1u || magic == 0x4d3cb2a1u);
    keep(&w, 0, 0); /* the last run */
    const int e = w.err ? errno : 0;
    if (fclose(f) != 0 || w.err) {
        const int e2 = e ? e : errno;
        unlink(out_path);
        kmpb_fail(KMPB_EIO, "%s: %s", out_path, strerror(e2));
        errno = e2;
        return KMPB_EIO;
    }
    if (n_written) *n_written = w.written;
    return KMPB_OK;
}
