/* dump_tables.c -- prints, one hex word per line, the host tables that decide the union engine's answers for a strings
 * file without windows: distinct count, pattern -> distinct id, the prefilter words, the probe tables (vtab) and the
 * prefix gate.  argv: <strings.txt> <flags mode: 0 none, 1 all nocase, 2 every third nocase> [win].  With "win" the
 * tables come from kmpb_tables_build_win with every window {0, KMPB_WINDOW_ANY}, else from kmpb_tables_build_flags.
 * tests/test_tables_windows.py hashes the output and compares it with tests/golden/tables_sha256.json, which holds the
 * hashes of the tables the library built before windows existed. */
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "kmpb_internal.h"

int main(int argc, char **argv)
{
    if (argc < 3) return 2;
    kmpb_patterns pats;
    if (kmpb_load_patterns_file(argv[1], &pats) != 0) return 2;
    const int mode = atoi(argv[2]);
    uint8_t *flags = calloc(pats.n_pat + 1, 1);
    for (uint32_t i = 0; i < pats.n_pat; i++) flags[i] = mode == 1 || (mode == 2 && i % 3 == 1) ? KMPB_PAT_NOCASE : 0;
    kmpb_tables t;
    int rc;
#ifdef KMPB_WINDOW_ANY
    if (argc > 3 && strcmp(argv[3], "win") == 0) {
        kmpb_window *win = malloc((pats.n_pat + 1) * sizeof *win);
        for (uint32_t i = 0; i < pats.n_pat; i++) { win[i].lo = 0; win[i].hi = KMPB_WINDOW_ANY; }
        rc = kmpb_tables_build_win(&t, pats.blob, pats.pat_off, pats.n_pat, flags, win, 0);
        free(win);
    } else
#endif
        rc = kmpb_tables_build_flags(&t, pats.blob, pats.pat_off, pats.n_pat, flags, 0);
    if (rc != 0) return 2;
    printf("%08x\n", t.n_uniq);
    for (uint32_t i = 0; i < t.n_pat; i++) printf("%08x\n", t.pat_to_uniq[i]);
    for (int c = 0; c < 256; c++) printf("%08x\n", t.filter6[c]);
    printf("%08x\n", t.vtab_words);
    for (uint32_t i = 0; i < t.vtab_words; i++) printf("%08x\n", t.vtab[i]);
    printf("%08x %08x\n", t.gate_words, t.gate_shift);
    for (uint32_t i = 0; i < t.gate_words; i++) printf("%08x\n", t.gate[i]);
    kmpb_tables_free(&t);
    kmpb_free_patterns(&pats);
    free(flags);
    return 0;
}
