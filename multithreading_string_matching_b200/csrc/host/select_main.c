/* select_main.c -- kmp_select: the frames of a savefile that hold a match, written to a new savefile.
 *
 *   kmp_select [-i] [-v] <file.pcap> <string.txt> <out.pcap> [udp|tcp]
 *
 * -i makes every token case-insensitive (ASCII letters, KMPB_PAT_NOCASE), as for kmp_find; -v writes the frames that
 * hold NO match instead (dropping known noise); -w LO:HI counts a token only where it starts at a payload offset in
 * [LO, HI] (cli_window.h).  The options come in any order before the file names.  A frame is selected when its UDP or TCP payload holds at least one
 * match that kmp_match counts, i.e. when kmp_find prints a line for it.  The output has the input's format (classic
 * or pcapng, byte order, timestamp resolution, link type) and holds the chosen records byte for byte; frames whose
 * payload the extractor refused are in neither output.  stdout is one line, "<selected> of <accepted> packets written
 * to <out.pcap>" (with -v, <selected> counts the frames written).  Usage text goes to stdout with exit status 1;
 * unreadable inputs and the missing B200 fail as in kmp_find.
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
    const char *prog = "./kmp_select";
    int proto = KMPB_PROTO_UDP, nocase = 0, invert = 0, windowed = 0;
    kmpb_window window;
    for (; argc > 1 && argv[1][0] == '-' && argv[1][1] && !argv[1][2]; argv++, argc--) {
        if (argv[1][1] == 'i') nocase = 1;
        else if (argv[1][1] == 'v') invert = 1;
        else if (argv[1][1] == 'w') {
            if (!parse_window_arg(argc > 2 ? argv[2] : NULL, &window)) return bad_window(argc > 2 ? argv[2] : NULL);
            windowed = 1;
            argv++;
            argc--;
        } else break;
    }
    if (argc < 4 || argc > 5) {
        printf("USAGE: %s [-i] [-v] <file.pcap> <string.txt> <out.pcap> [tcp/udp]\n", prog);
        return 1;
    }
    if (argc == 5) {
        if (strcmp(argv[4], "udp") == 0) proto = KMPB_PROTO_UDP;
        else if (strcmp(argv[4], "tcp") == 0) proto = KMPB_PROTO_TCP;
        else {
            printf("USAGE %s [-i] [-v] <file.pcap> <string.txt> <out.pcap> [tcp/udp]\n", prog);
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
    uint8_t *pflags = nocase ? malloc(pats.n_pat ? pats.n_pat : 1) : NULL;
    if (pflags) memset(pflags, KMPB_PAT_NOCASE, pats.n_pat);
    kmpb_window *win = window_array(windowed ? &window : NULL, pats.n_pat);
    if (windowed && win == NULL) return fail("out of memory");
    rc = kmpb_set_patterns_win(ctx, pats.blob, pats.pat_off, pats.n_pat, pflags, win);
    free(pflags);
    free(win);
    if (rc != 0) return fail("patterns");

    const uint64_t n_packets = kmpb_pcap_packets(pc);
    uint8_t *verdicts = malloc(n_packets ? n_packets : 1);
    if (verdicts == NULL) return fail("out of memory");
    uint64_t selected = 0, written = 0;
    if (kmpb_select_pcap(ctx, pc, 0, n_packets, verdicts, &selected, NULL) != 0) return fail("select");
    kmpb_destroy(ctx);
    if (kmpb_pcap_write_selected(pc, 0, n_packets, verdicts, invert, argv[3], &written) != 0) return fail("write");
    printf("%llu of %llu packets written to %s\n", (unsigned long long)written, (unsigned long long)n_packets, argv[3]);

    free(verdicts);
    kmpb_pcap_close(pc);
    kmpb_free_patterns(&pats);
    return 0;
}
