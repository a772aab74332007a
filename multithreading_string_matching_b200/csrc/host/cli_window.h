/* cli_window.h -- the -w LO:HI option of kmp_match, kmp_find and kmp_select: one position window for every token of
 * the strings file (kmpb_set_patterns_win), as -i gives every token the nocase flag.  LO and HI are decimal, with
 * 0 <= LO <= HI <= 65535 (KMPB_WINDOW_MAX).  The programs parse it before anything else runs; a malformed value is
 * "error: bad window ..." on stderr and exit status 1. */
#ifndef KMPB_CLI_WINDOW_H
#define KMPB_CLI_WINDOW_H

#include <stdio.h>
#include <stdlib.h>

#include "kmpb200.h"

/* 1 and *w set when s is LO:HI, else 0 */
static int parse_window_arg(const char *s, kmpb_window *w)
{
    uint32_t v[2];
    if (s == NULL) return 0;
    for (int k = 0; k < 2; k++) {
        const char *start = s;
        uint32_t x = 0;
        for (; *s >= '0' && *s <= '9'; s++)
            if ((x = 10 * x + (uint32_t)(*s - '0')) > KMPB_WINDOW_MAX) return 0;
        if (s == start) return 0;
        v[k] = x;
        if (k == 0 && *s++ != ':') return 0;
    }
    if (*s != '\0' || v[0] > v[1]) return 0;
    w->lo = v[0];
    w->hi = v[1];
    return 1;
}

static int bad_window(const char *s)
{
    fprintf(stderr, "error: bad window '%s': expected LO:HI, decimal, with 0 <= LO <= HI <= %u\n", s ? s : "", KMPB_WINDOW_MAX);
    return 1;
}

/* n copies of *w (NULL when w is NULL: no window) */
static kmpb_window *window_array(const kmpb_window *w, uint32_t n)
{
    if (w == NULL) return NULL;
    kmpb_window *a = malloc((n ? n : 1) * sizeof *a);
    if (a)
        for (uint32_t i = 0; i < n; i++) a[i] = *w;
    return a;
}

#endif
