/* find_main.c -- kmp_find: where the patterns of a strings file occur in a savefile, one line per match.
 *
 *   kmp_find <file.pcap> <string.txt> [udp|tcp]
 *   kmp_find -i <file.pcap> <string.txt> [udp|tcp]     every token case-insensitive (ASCII letters, KMPB_PAT_NOCASE)
 *   kmp_find -w LO:HI <file.pcap> <string.txt> ...     only the matches that start at a payload offset in [LO, HI]
 *                                                      (cli_window.h); -i and -w combine, in either order
 *
 * stdout: "<frame> <offset> <pattern>\n" per match, ordered by (frame, offset, pattern index): frame is the 1-based
 * capture record number (the numbering Wireshark shows), offset the position of the match's first byte inside the
 * frame's UDP or TCP payload, pattern the token as the strings file spells it (a token listed several times is
 * reported once per match, under its first listing).  The matches are exactly those kmp_match counts.  Usage text goes
 * to stdout with exit status 1; an unreadable strings file is perror("error opening file: ") + exit 1; an unreadable
 * pcap is "error reading pcap file: ..." on stderr + exit 1 -- as kmp_match does.
 */
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "cli_window.h"
#include "kmpb200.h"

static int fail(const char *what)
{
    fprintf(stderr, "error: %s: %s\n", what, kmpb_last_error());
    return 1;
}

int main(int argc, char **argv)
{
    const char *prog = "./kmp_find";
    int proto = KMPB_PROTO_UDP;
    /* -i and -w LO:HI, each at most once, in either order; then the arguments follow as without them */
    int nocase = 0, windowed = 0;
    kmpb_window window;
    for (int k = 0; k < 2 && argc > 1; k++) {
        if (!nocase && strcmp(argv[1], "-i") == 0) nocase = 1;
        else if (!windowed && strcmp(argv[1], "-w") == 0) {
            if (!parse_window_arg(argc > 2 ? argv[2] : NULL, &window)) return bad_window(argc > 2 ? argv[2] : NULL);
            windowed = 1;
            argv++;
            argc--;
        } else break;
        argv++;
        argc--;
    }
    if (argc < 3 || argc > 4) {
        printf("USAGE: %s <file.pcap> <string.txt> [tcp/udp]\n", prog);
        return 1;
    }
    if (argc == 4) {
        if (strcmp(argv[3], "udp") == 0) proto = KMPB_PROTO_UDP;
        else if (strcmp(argv[3], "tcp") == 0) proto = KMPB_PROTO_TCP;
        else {
            printf("USAGE %s <file.pcap> <string.txt> [tcp/udp]\n", prog);
            return 1;
        }
    }

    kmpb_patterns pats;
    int rc = kmpb_load_patterns_file(argv[2], &pats);
    if (rc == KMPB_EIO) {
        perror("error opening file: ");
        return 1;
    }
    if (rc != 0) {
        fprintf(stderr, "error reading patterns: %s\n", kmpb_last_error());
        return 1;
    }
    if (kmpb_device_count() <= 0) {
        fprintf(stderr, "error: no B200-class CUDA device available (this program has no CPU path)\n");
        return 1;
    }
    kmpb_pcap *pc = NULL;
    if (kmpb_pcap_open(argv[1], proto, &pc) != 0) {
        fprintf(stderr, "error reading pcap file: %s\n", kmpb_last_error());
        return 1;
    }
    kmpb_ctx *ctx = NULL;
    if (kmpb_create(&ctx, kmpb_device_ordinal(0)) != 0) return fail("GPU");
    uint8_t *flags = nocase ? malloc(pats.n_pat ? pats.n_pat : 1) : NULL;
    if (flags) memset(flags, KMPB_PAT_NOCASE, pats.n_pat);
    kmpb_window *win = window_array(windowed ? &window : NULL, pats.n_pat);
    if (windowed && win == NULL) return fail("out of memory");
    rc = kmpb_set_patterns_win(ctx, pats.blob, pats.pat_off, pats.n_pat, flags, win);
    free(flags);
    free(win);
    if (rc != 0) return fail("patterns");

    /* a guess first (C3-like traffic has one match per ~400 payload bytes), then the exact size if it was short */
    const uint64_t n_packets = kmpb_pcap_packets(pc);
    uint64_t capacity = kmpb_pcap_bytes(pc) / 256 + 4096, total = 0;
    kmpb_match *m = malloc(capacity * sizeof *m);
    if (m == NULL) return fail("out of memory");
    if (kmpb_find_pcap(ctx, pc, 0, n_packets, m, capacity, &total) != 0) return fail("find");
    if (total > capacity) {
        free(m);
        capacity = total;
        m = malloc(capacity * sizeof *m);
        if (m == NULL) return fail("out of memory");
        if (kmpb_find_pcap(ctx, pc, 0, n_packets, m, capacity, &total) != 0) return fail("find");
    }
    uint64_t *frames = malloc((n_packets ? n_packets : 1) * sizeof *frames);
    if (frames == NULL) return fail("out of memory");
    if (kmpb_pcap_frame_index(pc, 0, n_packets, frames) != 0) return fail("frames");

    static char obuf[1 << 20];
    setvbuf(stdout, obuf, _IOFBF, sizeof obuf);
    for (uint64_t i = 0; i < total; i++) {
        const uint32_t p = m[i].pattern;
        printf("%llu %u ", (unsigned long long)frames[m[i].packet] + 1ull, m[i].offset);
        fwrite(pats.blob + pats.pat_off[p], 1, pats.pat_off[p + 1] - pats.pat_off[p], stdout);
        putchar('\n');
    }
    fflush(stdout);

    free(frames);
    free(m);
    kmpb_destroy(ctx);
    kmpb_pcap_close(pc);
    kmpb_free_patterns(&pats);
    return 0;
}
