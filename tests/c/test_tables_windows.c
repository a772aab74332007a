/* test_tables_windows.c -- CPU check of the host-built tables for pattern sets with position windows
 * (csrc/host/automaton.c kmpb_tables_build_win), no GPU involved.
 *
 *   1. a set without windows (win NULL, or every window {0, KMPB_WINDOW_ANY}) builds word for word the tables
 *      kmpb_tables_build_flags builds: ids, filter, probe tables, gate, and no window tables (that those are the tables
 *      of the library before windows is checked against stored hashes: tests/c/dump_tables.c);
 *   2. in a seeded random mixed set, the union engine's tables (filter, probe tables, gate, n_nocase) equal those of its
 *      unwindowed subset built alone, and the unwindowed patterns keep that subset's ids;  the windowed distinct
 *      patterns follow them, one per (bytes, flag, window), with their windows, the reach max(hi + len) and the first
 *      bytes they can start with; every windowed pattern finds its record under its own id in the window probe table;
 *   3. every invalid window is KMPB_EINVAL naming the pattern.
 * Exit status 0 = all good.  Built and run by tests/test_tables_windows.py.
 */
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "kmpb_internal.h"

static uint64_t rng_state = 0x2545f4914f6cdd1dull;
static uint32_t rnd(void)
{
    rng_state ^= rng_state << 13; rng_state ^= rng_state >> 7; rng_state ^= rng_state << 17;
    return (uint32_t)(rng_state >> 11);
}

static int bad = 0;
#define CHECK(cond, ...)                                                                                              \
    do {                                                                                                              \
        if (!(cond)) { fprintf(stderr, __VA_ARGS__); fputc('\n', stderr); bad = 1; return; }                          \
    } while (0)

static int same_union_tables(const kmpb_tables *a, const kmpb_tables *b)
{
    return a->n_union == b->n_union && a->n_nocase == b->n_nocase && a->vtab_words == b->vtab_words &&
           memcmp(a->vtab, b->vtab, 4ull * a->vtab_words) == 0 && memcmp(a->filter6, b->filter6, sizeof a->filter6) == 0 &&
           a->gate_words == b->gate_words && a->gate_shift == b->gate_shift &&
           (a->gate_words == 0 || memcmp(a->gate, b->gate, 4ull * a->gate_words) == 0);
}

/* the probe-table record of distinct id u in table v (the way the device probes: key slot, then the slot's records); a
 * one-byte pattern: the table's id starts a run down to u of the same byte and flag (window.cu window_probe) */
static int has_record(const kmpb_tables *t, const uint32_t *v, const uint8_t *p, uint32_t len, uint32_t nc, uint32_t u)
{
    if (len == 1) {
        const uint32_t top = v[v[5] + (nc ? 256u : 0u) + p[0]];
        if (top == 0xffffffffu || top < u) return 0;
        for (uint32_t w = u; w <= top; w++)
            if (t->uniq_len[w] != 1 || t->uniq_blob[t->uniq_off[w]] != p[0] || t->uniq_flags[w] != nc) return 0;
        return 1;
    }
    const uint32_t key = len >= 3 ? (p[0] | (uint32_t)p[1] << 8 | (uint32_t)p[2] << 16) : (p[0] | (uint32_t)p[1] << 8);
    const uint32_t so = len >= 3 ? v[3] : v[1], sh = len >= 3 ? v[4] : v[2];
    const uint32_t s = kmpb_vtab_slot(key, sh);
    for (uint32_t j = 0; j < v[so + 2 * s + 1]; j++) {
        const uint32_t *rec = v + v[6] + 8 * (v[so + 2 * s] + j);
        if (rec[5] == u && rec[4] == len) return 1;
    }
    return 0;
}

static void without_windows(void)
{
    const char *toks[] = {"GET", "get", "a", "ab", "http", "abcdefghijk", "GET", "Host:", "zz"};
    const uint32_t n = sizeof toks / sizeof *toks;
    uint8_t blob[256], flags[16];
    uint32_t off[16], at = 0;
    kmpb_window win[16];
    for (uint32_t i = 0; i < n; i++) {
        off[i] = at;
        memcpy(blob + at, toks[i], strlen(toks[i]));
        at += (uint32_t)strlen(toks[i]);
        flags[i] = i % 3 == 1 ? KMPB_PAT_NOCASE : 0;
        win[i].lo = 0;
        win[i].hi = KMPB_WINDOW_ANY;
    }
    off[n] = at;
    kmpb_tables a, b, c;
    CHECK(kmpb_tables_build_flags(&a, blob, off, n, flags, 0) == 0, "build_flags: %s", kmpb_last_error());
    CHECK(kmpb_tables_build_win(&b, blob, off, n, flags, NULL, 0) == 0, "build_win NULL: %s", kmpb_last_error());
    CHECK(kmpb_tables_build_win(&c, blob, off, n, flags, win, 0) == 0, "build_win any: %s", kmpb_last_error());
    const kmpb_tables *t[2] = {&b, &c};
    for (int k = 0; k < 2; k++) {
        CHECK(same_union_tables(&a, t[k]) && t[k]->n_uniq == a.n_uniq && t[k]->n_union == a.n_uniq, "tables differ (%d)", k);
        CHECK(memcmp(a.pat_to_uniq, t[k]->pat_to_uniq, 4ull * n) == 0, "ids differ (%d)", k);
        CHECK(t[k]->wvtab == NULL && t[k]->wvtab_words == 0 && t[k]->win_reach == 0, "window tables without windows (%d)", k);
    }
    kmpb_tables_free(&a);
    kmpb_tables_free(&b);
    kmpb_tables_free(&c);
}

static void mixed_sets(void)
{
    const char *alpha = "abcAB@";
    for (int trial = 0; trial < 300; trial++) {
        const uint32_t n = 1 + rnd() % 24;
        uint8_t blob[24 * 12], flags[24], sub_blob[24 * 12], sub_flags[24];
        uint32_t off[25], sub_off[25], sub_of[24], at = 0, ns = 0, sat = 0;
        kmpb_window win[24];
        for (uint32_t i = 0; i < n; i++) {
            off[i] = at;
            uint32_t len = 1 + rnd() % 11;
            if (i > 0 && rnd() % 4 == 0) { /* an earlier pattern again, maybe with another window or flag */
                const uint32_t j = rnd() % i;
                len = off[j + 1] - off[j];
                memcpy(blob + at, blob + off[j], len);
            } else {
                for (uint32_t k = 0; k < len; k++) blob[at + k] = (uint8_t)alpha[rnd() % 6];
            }
            at += len;
            flags[i] = rnd() % 3 == 0 ? KMPB_PAT_NOCASE : 0;
            const uint32_t lo = rnd() % 3 == 0 ? rnd() % 70000 % (KMPB_WINDOW_MAX + 1) : rnd() % 8;
            if (rnd() % 2) { win[i].lo = 0; win[i].hi = KMPB_WINDOW_ANY; }
            else { win[i].lo = lo; win[i].hi = lo + rnd() % (KMPB_WINDOW_MAX + 1 - lo); }
            if (win[i].hi == KMPB_WINDOW_ANY) { /* the unwindowed subset */
                sub_off[ns] = sat;
                memcpy(sub_blob + sat, blob + off[i], len);
                sat += len;
                sub_flags[ns] = flags[i];
                sub_of[ns++] = i;
            }
        }
        off[n] = at;
        sub_off[ns] = sat;
        kmpb_tables t, s;
        CHECK(kmpb_tables_build_win(&t, blob, off, n, flags, win, 1) == 0, "build mixed: %s", kmpb_last_error());
        CHECK(kmpb_tables_build_flags(&s, sub_blob, sub_off, ns, sub_flags, 1) == 0, "build subset: %s", kmpb_last_error());
        CHECK(same_union_tables(&t, &s), "trial %d: union tables differ from the unwindowed subset's", trial);
        CHECK(t.n_state == s.n_state && memcmp(t.next, s.next, 4ull * s.n_state * s.n_class) == 0, "trial %d: automaton", trial);
        for (uint32_t j = 0; j < ns; j++) CHECK(t.pat_to_uniq[sub_of[j]] == s.pat_to_uniq[j], "trial %d: id of pattern %u", trial, sub_of[j]);
        /* windowed distinct patterns: one per (bytes, flag, window), after the others */
        uint32_t reach = 0, first[8] = {0};
        for (uint32_t i = 0; i < n; i++) {
            if (win[i].hi == KMPB_WINDOW_ANY) continue;
            const uint32_t u = t.pat_to_uniq[i], w = u - t.n_union, len = off[i + 1] - off[i];
            CHECK(u >= t.n_union && u < t.n_uniq, "trial %d: windowed pattern %u has id %u", trial, i, u);
            CHECK(t.uniq_lo[w] == win[i].lo && t.uniq_hi[w] == win[i].hi, "trial %d: window of pattern %u", trial, i);
            CHECK(has_record(&t, t.wvtab, t.uniq_blob + t.uniq_off[u], len, flags[i], u), "trial %d: no record of %u", trial, i);
            for (uint32_t j = 0; j < i; j++) {
                const int same = off[j + 1] - off[j] == len && flags[j] == flags[i] && win[j].lo == win[i].lo &&
                                 win[j].hi == win[i].hi &&
                                 (flags[i] ? strncasecmp((const char *)blob + off[j], (const char *)blob + off[i], len) == 0
                                           : memcmp(blob + off[j], blob + off[i], len) == 0);
                CHECK(same == (t.pat_to_uniq[j] == u), "trial %d: patterns %u and %u", trial, j, i);
            }
            if (win[i].hi + len > reach) reach = win[i].hi + len;
            uint8_t c = blob[off[i]];
            first[c >> 5] |= 1u << (c & 31);
            if (flags[i] && ((c | 0x20) >= 'a' && (c | 0x20) <= 'z')) first[(c ^ 0x20) >> 5] |= 1u << ((c ^ 0x20) & 31);
        }
        CHECK(t.win_reach == reach && memcmp(t.win_first, first, sizeof first) == 0, "trial %d: reach / first bytes", trial);
        kmpb_tables_free(&t);
        kmpb_tables_free(&s);
    }
}

static void invalid_windows(void)
{
    const uint8_t blob[] = "abcdef";
    const uint32_t off[] = {0, 2, 4, 6};
    const kmpb_window bad_windows[][2] = {
        {{5, 4}, {0, 0}},                         /* lo > hi */
        {{0, KMPB_WINDOW_MAX + 1}, {0, 0}},       /* hi above the limit */
        {{1, KMPB_WINDOW_ANY}, {0, 0}},           /* open at the top */
        {{KMPB_WINDOW_ANY, KMPB_WINDOW_ANY}, {0, 0}},
    };
    for (size_t k = 0; k < sizeof bad_windows / sizeof *bad_windows; k++) {
        kmpb_window win[3] = {{0, KMPB_WINDOW_ANY}, bad_windows[k][0], bad_windows[k][1]};
        kmpb_tables t;
        CHECK(kmpb_tables_build_win(&t, blob, off, 3, NULL, win, 0) == KMPB_EINVAL && strstr(kmpb_last_error(), "pattern 1"),
              "window %zu accepted or not named: %s", k, kmpb_last_error());
    }
    kmpb_window ok[3] = {{0, KMPB_WINDOW_ANY}, {0, KMPB_WINDOW_MAX}, {KMPB_WINDOW_MAX, KMPB_WINDOW_MAX}};
    kmpb_tables t;
    CHECK(kmpb_tables_build_win(&t, blob, off, 3, NULL, ok, 0) == 0, "valid windows refused: %s", kmpb_last_error());
    CHECK(t.n_union == 1 && t.n_uniq == 3 && t.win_lo_min == 0 && t.win_hi_max == KMPB_WINDOW_MAX &&
          t.win_reach == KMPB_WINDOW_MAX + 2, "extremes of the windows");
    kmpb_tables_free(&t);
}

int main(void)
{
    without_windows();
    mixed_sets();
    invalid_windows();
    if (!bad) printf("test_tables_windows: ok\n");
    return bad;
}
