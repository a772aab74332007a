/* window_geometry.c -- prints "n_pat n_uniq n_union wvtab_words" of the tables kmpb_tables_build_win builds for a
 * pattern set with per-pattern flags and windows: what decides where the window kernel (csrc/cuda/window.cu) keeps its
 * counters (shared memory for at most 4096 distinct windowed patterns) and its probe tables (shared memory for at most
 * 16384 words).  argv: <set file>, one pattern a line: "<flags> <lo> <hi> <bytes in hex>", decimal numbers, hi
 * 4294967295 (KMPB_WINDOW_ANY) with lo 0 for no window.  tests/test_windows_scale.py writes the sets and checks which
 * path each of its cases takes. */
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "kmpb_internal.h"

int main(int argc, char **argv)
{
    if (argc < 2) return 2;
    FILE *f = fopen(argv[1], "r");
    if (!f) return 2;
    uint32_t cap = 1024, n = 0;
    uint8_t *flags = malloc(cap), *blob = malloc((size_t)cap * KMPB_MAX_PATTERN_LEN);
    uint32_t *off = malloc(((size_t)cap + 1) * sizeof *off);
    kmpb_window *win = malloc((size_t)cap * sizeof *win);
    char hex[2 * KMPB_MAX_PATTERN_LEN + 2];
    unsigned fl, lo, hi;
    off[0] = 0;
    while (fscanf(f, "%u %u %u %200s", &fl, &lo, &hi, hex) == 4) {
        if (n == cap) {
            cap *= 2;
            flags = realloc(flags, cap);
            blob = realloc(blob, (size_t)cap * KMPB_MAX_PATTERN_LEN);
            off = realloc(off, ((size_t)cap + 1) * sizeof *off);
            win = realloc(win, (size_t)cap * sizeof *win);
        }
        const size_t len = strlen(hex) / 2;
        if (len == 0 || len > KMPB_MAX_PATTERN_LEN || strlen(hex) % 2) return 2;
        for (size_t k = 0; k < len; k++) {
            unsigned b;
            if (sscanf(hex + 2 * k, "%2x", &b) != 1) return 2;
            blob[off[n] + k] = (uint8_t)b;
        }
        off[n + 1] = off[n] + (uint32_t)len;
        flags[n] = (uint8_t)fl;
        win[n].lo = lo;
        win[n].hi = hi;
        n++;
    }
    fclose(f);
    kmpb_tables t;
    if (kmpb_tables_build_win(&t, blob, off, n, flags, win, 0) != 0) {
        fprintf(stderr, "%s\n", kmpb_last_error());
        return 1;
    }
    printf("%u %u %u %u\n", t.n_pat, t.n_uniq, t.n_union, t.wvtab_words);
    kmpb_tables_free(&t);
    free(flags); free(blob); free(off); free(win);
    return 0;
}
