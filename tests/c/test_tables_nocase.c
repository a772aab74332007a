/* test_tables_nocase.c -- CPU check of the host-built tables for pattern sets with KMPB_PAT_NOCASE patterns
 * (csrc/host/automaton.c kmpb_tables_build_flags), no GPU involved.
 *
 *   1. all-zero flags build word for word the tables kmpb_tables_build builds (filter, probe tables, gate);
 *   2. on seeded random mixed sets over alphabets rich in letters and in the non-letter bytes that differ from another
 *      byte in bit 5 only (@ `, [ {, \ |, ] }, ^ ~, _ DEL, 0xC1 0xE1, 0xDF 0xFF):
 *      - every case variant of every nocase pattern's start passes the prefilter and the prefix gate;
 *      - every case variant of its key finds the pattern's record in the probe table;
 *      - the record's masked compare (first 8 bytes) and its tail masks accept exactly the case variants;
 *      - the probe tables, probed the way the device probes them, and the merged DFA count what a naive folded
 *        counter counts on random text.
 * Exit status 0 = all good.  Built and run by tests/test_tables_nocase.py.
 */
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "kmpb_internal.h"

static uint64_t rng_state = 0x9e3779b97f4a7c15ull;
static uint32_t rnd(void)
{
    rng_state ^= rng_state << 13; rng_state ^= rng_state >> 7; rng_state ^= rng_state << 17;
    return (uint32_t)(rng_state >> 11);
}

static uint8_t fold(uint8_t c) { return c >= 'A' && c <= 'Z' ? (uint8_t)(c + 32) : c; }
static int is_letter(uint8_t c) { return (c | 0x20) >= 'a' && (c | 0x20) <= 'z'; }
static int same_byte(int nc, uint8_t a, uint8_t b) { return nc ? fold(a) == fold(b) : a == b; }

static int bad = 0;
#define CHECK(cond, ...)                                                                                              \
    do {                                                                                                              \
        if (!(cond)) { fprintf(stderr, __VA_ARGS__); fputc('\n', stderr); bad = 1; return; }                          \
    } while (0)

static void random_set(int n_pat, int max_len, const char *alpha, uint8_t *blob, uint32_t *off, uint8_t *flags, int nc_mode)
{
    const int na = (int)strlen(alpha);
    uint32_t at = 0;
    for (int i = 0; i < n_pat; i++) {
        off[i] = at;
        int len = 1 + (int)(rnd() % (uint32_t)max_len);
        if (i > 0 && rnd() % 6 == 0) { /* an earlier pattern again, its letters' case flipped at random */
            int j = (int)(rnd() % (uint32_t)i);
            len = (int)(off[j + 1] - off[j]);
            for (int k = 0; k < len; k++) {
                uint8_t c = blob[off[j] + k];
                blob[at + k] = is_letter(c) && rnd() % 2 ? c ^ 0x20 : c;
            }
        } else {
            for (int k = 0; k < len; k++) blob[at + k] = (uint8_t)alpha[rnd() % (uint32_t)na];
        }
        flags[i] = nc_mode == 0 ? 0 : nc_mode == 1 ? KMPB_PAT_NOCASE : (rnd() % 2 ? KMPB_PAT_NOCASE : 0);
        at += (uint32_t)len;
    }
    off[n_pat] = at;
}

/* 1. all-zero flags: the tables of kmpb_tables_build, word for word */
static void zero_flags_identical(int n_pat, int max_len, const char *alpha)
{
    uint8_t *blob = malloc((size_t)n_pat * 99 + 1), *flags = calloc((size_t)n_pat + 1, 1);
    uint32_t *off = malloc(((size_t)n_pat + 1) * sizeof *off);
    random_set(n_pat, max_len, alpha, blob, off, flags, 0);
    kmpb_tables a, b;
    CHECK(kmpb_tables_build(&a, blob, off, (uint32_t)n_pat) == 0, "build: %s", kmpb_last_error());
    CHECK(kmpb_tables_build_flags(&b, blob, off, (uint32_t)n_pat, flags, 0) == 0, "build_flags: %s", kmpb_last_error());
    CHECK(a.n_uniq == b.n_uniq && b.n_nocase == 0, "distinct patterns differ");
    CHECK(memcmp(a.pat_to_uniq, b.pat_to_uniq, (size_t)n_pat * 4) == 0, "pattern map differs");
    CHECK(memcmp(a.filter6, b.filter6, sizeof a.filter6) == 0, "filter6 differs");
    CHECK(a.vtab_words == b.vtab_words && memcmp(a.vtab, b.vtab, (size_t)a.vtab_words * 4) == 0, "vtab differs");
    CHECK(a.gate_words == b.gate_words && a.gate_shift == b.gate_shift &&
              (a.gate_words == 0 || memcmp(a.gate, b.gate, (size_t)a.gate_words * 4) == 0), "gate differs");
    kmpb_tables_free(&a);
    kmpb_tables_free(&b);
    free(blob); free(flags); free(off);
}

/* the variant of the folded pattern p whose letters among bytes [0, n) take the case bits of `bits` */
static void variant(const uint8_t *p, uint32_t len, int nc, uint32_t n, uint32_t bits, uint8_t *out)
{
    memcpy(out, p, len);
    for (uint32_t i = 0, k = 0; i < n && i < len; i++)
        if (nc && is_letter(p[i])) out[i] = (bits >> k++) & 1 ? (uint8_t)(p[i] ^ 0x20) : p[i];
}

static void mixed_case(int n_pat, int max_len, const char *alpha, int text_len, int nc_mode)
{
    uint8_t *blob = malloc((size_t)n_pat * 99 + 1), *flags = calloc((size_t)n_pat + 1, 1);
    uint32_t *off = malloc(((size_t)n_pat + 1) * sizeof *off);
    random_set(n_pat, max_len, alpha, blob, off, flags, nc_mode);
    const int na = (int)strlen(alpha);
    uint8_t *text = calloc((size_t)text_len + 16, 1);
    for (int i = 0; i < text_len; i++) text[i] = (uint8_t)alpha[rnd() % (uint32_t)na];
    for (int r = 0; r < 8 && n_pat; r++) { /* plant case variants */
        int p = (int)(rnd() % (uint32_t)n_pat), len = (int)(off[p + 1] - off[p]);
        if (len >= text_len) continue;
        uint8_t *dst = text + rnd() % (uint32_t)(text_len - len);
        for (int k = 0; k < len; k++) {
            uint8_t c = blob[off[p] + k];
            dst[k] = flags[p] && is_letter(c) && rnd() % 2 ? c ^ 0x20 : c;
        }
    }

    kmpb_tables t;
    CHECK(kmpb_tables_build_flags(&t, blob, off, (uint32_t)n_pat, flags, 1) == 0, "build failed: %s", kmpb_last_error());
    const uint32_t *v = t.vtab;
    uint8_t w[128];

    /* distinct patterns: (folded bytes, flag) */
    for (int p = 0; p < n_pat; p++) {
        const uint32_t u = t.pat_to_uniq[p], len = off[p + 1] - off[p];
        CHECK(t.uniq_len[u] == len && t.uniq_flags[u] == flags[p], "pattern %d: wrong distinct pattern", p);
        for (uint32_t k = 0; k < len; k++)
            CHECK(t.uniq_blob[t.uniq_off[u] + k] == (flags[p] ? fold(blob[off[p] + k]) : blob[off[p] + k]), "pattern %d: stored bytes", p);
    }

    for (uint32_t u = 0; u < t.n_uniq; u++) {
        const uint8_t *p = t.uniq_blob + t.uniq_off[u];
        const uint32_t len = t.uniq_len[u], nc = t.uniq_flags[u];
        uint32_t nl = 0;
        for (uint32_t i = 0; i < len && i < 4; i++) nl += nc && is_letter(p[i]);
        for (uint32_t bits = 0; bits < (1u << nl); bits++) {
            variant(p, len, (int)nc, 4, bits, w);
            w[len] = w[len + 1] = w[len + 2] = w[len + 3] = 0;
            /* the prefilter: the start's report after its fourth byte (text zero padded) */
            uint32_t S = 0;
            for (int k = 0; k < 4; k++) S = ((S << 6) | 0x3fu) & t.filter6[w[k]];
            CHECK(S & (0x1fu << 18), "filter6 misses a variant of uniq %u", u);
            /* the gate */
            if (t.gate_words) {
                const uint32_t g = t.gate[kmpb_gate_slot(w[0] | (uint32_t)w[1] << 8, t.gate_shift)];
                CHECK(len < 3 ? g == 0xffffffffu : (g >> (31 - (w[2] & 31))) & 1u, "gate rejects a variant of uniq %u", u);
            }
            if (len < 2) continue;
            /* the probe table: a record of u in the variant's slot */
            const uint32_t tab = len >= 3, so = v[1 + 2 * tab], shift = v[2 + 2 * tab];
            const uint32_t key = (uint32_t)w[0] | (uint32_t)w[1] << 8 | (tab ? (uint32_t)w[2] << 16 : 0u);
            const uint32_t *e = v + so + 2 * kmpb_vtab_slot(key, shift);
            int found = 0;
            for (uint32_t r = 0; r < e[1]; r++) found += v[v[6] + 8 * (e[0] + r) + 5] == u;
            CHECK(found == 1, "uniq %u: %d records in a variant's slot", u, found);
            /* the record accepts exactly the case variants, byte by byte */
            const uint32_t *rec = NULL;
            for (uint32_t r = 0; r < e[1]; r++)
                if (v[v[6] + 8 * (e[0] + r) + 5] == u) rec = v + v[6] + 8 * (e[0] + r);
            CHECK(rec[4] == len && (rec[7] != 0) == (nc && len > 8), "uniq %u: record words", u);
            if (bits) continue;
            for (uint32_t i = 0; i < len; i++)
                for (uint32_t c = 0; c < 256; c++) {
                    const uint32_t mword = i < 8 ? rec[1 + 2 * (i / 4)] : rec[7] ? v[rec[7] + i / 4] : 0xffffffffu;
                    const uint32_t pbyte = ((const uint8_t *)(v + v[7] + rec[6]))[i];
                    const uint32_t m = (mword >> (8 * (i % 4))) & 0xffu;
                    CHECK(((c ^ pbyte) & m) == 0 ? same_byte((int)nc, (uint8_t)c, p[i]) : !same_byte((int)nc, (uint8_t)c, p[i]),
                          "uniq %u byte %u: mask accepts 0x%02x wrongly", u, i, c);
                }
        }
    }

    /* counts: naive (folded for nocase), the probe tables as the device probes them, the merged DFA */
    uint64_t *naive = calloc((size_t)t.n_uniq + 1, 8), *probe = calloc((size_t)t.n_uniq + 1, 8), *dfa = calloc((size_t)t.n_uniq + 1, 8);
    for (uint32_t u = 0; u < t.n_uniq; u++) {
        const uint8_t *p = t.uniq_blob + t.uniq_off[u];
        const uint32_t len = t.uniq_len[u];
        for (int i = 0; i + (int)len <= text_len; i++) {
            uint32_t k = 0;
            while (k < len && same_byte(t.uniq_flags[u], text[i + k], p[k])) k++;
            naive[u] += k == len;
        }
    }
    for (int s = 0; s < text_len; s++) {
        uint32_t x0 = 0, x1 = 0;
        for (int k = 0; k < 4; k++) x0 |= (uint32_t)text[s + k] << (8 * k);
        for (int k = 0; k < 4; k++) x1 |= (uint32_t)text[s + 4 + k] << (8 * k);
        if (v[5]) {
            if (v[v[5] + (x0 & 0xffu)] != 0xffffffffu) probe[v[v[5] + (x0 & 0xffu)]]++;
            if (t.n_nocase && v[v[5] + 256 + (x0 & 0xffu)] != 0xffffffffu) probe[v[v[5] + 256 + (x0 & 0xffu)]]++;
        }
        for (int tab = 0; tab < 2; tab++) {
            const uint32_t so = v[1 + 2 * tab], shift = v[2 + 2 * tab];
            if (!so) continue;
            const uint32_t *e = v + so + 2 * kmpb_vtab_slot(x0 & (tab ? 0xffffffu : 0xffffu), shift);
            for (uint32_t r = 0; r < e[1]; r++) {
                const uint32_t *rec = v + v[6] + 8 * (e[0] + r);
                const uint32_t len = rec[4];
                if (((x0 ^ rec[0]) & rec[1]) | ((x1 ^ rec[2]) & rec[3])) continue;
                if (s + (int)len > text_len) continue;
                int same = 1;
                for (uint32_t jj = 8; jj < len && same; jj += 4) {
                    uint32_t tw = 0;
                    for (int k = 0; k < 4; k++) tw |= (uint32_t)text[s + jj + k] << (8 * k);
                    uint32_t diff = tw ^ v[v[7] + rec[6] + jj / 4];
                    if (rec[7]) diff &= v[rec[7] + jj / 4];
                    same = (len - jj >= 4 ? diff : diff & ((1u << (8 * (len - jj))) - 1u)) == 0;
                }
                probe[rec[5]] += same;
            }
        }
    }
    uint32_t state = 0;
    for (int i = 0; i < text_len; i++) {
        const uint32_t e = t.next[(size_t)state * t.n_class + t.byte_class[text[i]]];
        state = e & 0x7fffffffu;
        CHECK((e >> 31) == (t.out_head[state + 1] > t.out_head[state]), "report flag wrong");
        for (uint32_t o = t.out_head[state]; o < t.out_head[state + 1]; o++) dfa[t.out_id[o]]++;
    }
    for (uint32_t u = 0; u < t.n_uniq; u++)
        CHECK(probe[u] == naive[u] && dfa[u] == naive[u], "uniq %u (nocase %u, %u bytes): naive %llu probe %llu dfa %llu", u,
              t.uniq_flags[u], t.uniq_len[u], (unsigned long long)naive[u], (unsigned long long)probe[u], (unsigned long long)dfa[u]);
    free(naive); free(probe); free(dfa);
    kmpb_tables_free(&t);
    free(blob); free(flags); free(off); free(text);
}

int main(void)
{
    const char *alphas[] = {"aAbB", "abcABC@`[{", "aAbBzZ@`[{\\|]}^~_\x7f\xc1\xe1\xdf\xff",
                            "abcdefghijklmnopqrstuvwxyzABCDEFGHIJKLMNOPQRSTUVWXYZ0123456789-/:", "xX-_ .:/"};
    for (int trial = 0; trial < 64 && !bad; trial++) {
        const int n_pat = (int[]){1, 2, 5, 8, 30, 97, 300, 1200}[trial % 8];
        const int max_len = (int[]){1, 2, 3, 4, 8, 12, 40, 99}[(trial / 8) % 8];
        zero_flags_identical(n_pat, max_len, alphas[trial % 5]);
    }
    for (int trial = 0; trial < 240 && !bad; trial++) {
        const int n_pat = (int[]){1, 2, 3, 5, 8, 20, 40, 97}[trial % 8];
        const int max_len = (int[]){1, 2, 3, 4, 5, 9, 17, 40, 99, 12}[(trial / 8) % 10];
        mixed_case(n_pat, max_len, alphas[trial % 5], 200 + (int)(rnd() % 2000), 1 + trial % 3 % 2 + (trial % 3 == 2));
    }
    /* unknown flag bits are refused, naming the pattern */
    kmpb_tables t;
    const uint8_t blob[] = "abcd";
    const uint32_t off[] = {0, 2, 4};
    const uint8_t fl[] = {KMPB_PAT_NOCASE, 2};
    if (kmpb_tables_build_flags(&t, blob, off, 2, fl, 0) != KMPB_EINVAL || !strstr(kmpb_last_error(), "pattern 1")) {
        fprintf(stderr, "unknown flag accepted\n");
        bad = 1;
    }
    printf(bad ? "FAIL\n" : "OK\n");
    return bad;
}
