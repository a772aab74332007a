/* kmp_find_ref.c -- reference for the find tests (tests/test_find.py compiles it): where the matches that the oracle's
 * orc_count_csr counts are.  A restatement of kmp_matcher (serial.c:190-215) that records the start i - m + 1 of every
 * hit instead of counting it, on the text of each packet (serial.c:191: up to its first NUL byte).  A pattern equal to
 * an earlier one is not searched again: its matches are reported once, under the lowest index of the equal patterns.
 * Records {packet, offset, pattern} come sorted by (packet, offset, pattern); the first min(total, capacity) are
 * written.  Returns the total.  Test infrastructure only: the product never links it. */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

typedef struct { uint32_t offset, pattern; } hit;

static int hit_cmp(const void *a, const void *b)
{
    const hit *x = a, *y = b;
    if (x->offset != y->offset) return x->offset < y->offset ? -1 : 1;
    return x->pattern < y->pattern ? -1 : x->pattern > y->pattern;
}

/* serial.c:217-238 */
static void kmp_prefix(const unsigned char *p, int m, int *pi)
{
    int border = 0;
    pi[0] = 0;
    for (int i = 1; i < m; i++) {
        while (border > 0 && p[i] != p[border]) border = pi[border - 1];
        if (p[i] == p[border]) border++;
        pi[i] = border;
    }
}

int64_t kmpo_find_csr(const unsigned char *bytes, const uint64_t *offsets, uint64_t n_packets,
                      const unsigned char *pat_blob, const uint32_t *pat_off, uint32_t n_pat,
                      uint64_t *packet, uint32_t *offset, uint32_t *pattern, int64_t capacity)
{
    if (n_pat == 0) return 0;
    uint32_t *first = malloc((size_t)n_pat * sizeof *first), n_first = 0;
    int **pi = calloc(n_pat, sizeof *pi);
    for (uint32_t p = 0; p < n_pat; p++) {
        const uint32_t m = pat_off[p + 1] - pat_off[p];
        int dup = 0;
        for (uint32_t q = 0; q < n_first && !dup; q++)
            dup = pat_off[first[q] + 1] - pat_off[first[q]] == m && memcmp(pat_blob + pat_off[first[q]], pat_blob + pat_off[p], m) == 0;
        if (dup || m == 0) continue;
        first[n_first++] = p;
        pi[p] = malloc((size_t)m * sizeof(int));
        kmp_prefix(pat_blob + pat_off[p], (int)m, pi[p]);
    }
    size_t cap = 256, n = 0;
    hit *hits = malloc(cap * sizeof *hits);
    int64_t total = 0;
    for (uint64_t k = 0; k < n_packets; k++) {
        const unsigned char *text = bytes + offsets[k];
        const size_t plen = (size_t)(offsets[k + 1] - offsets[k]);
        const unsigned char *z = plen ? memchr(text, 0, plen) : NULL;
        const int64_t len = z ? (int64_t)(z - text) : (int64_t)plen;
        n = 0;
        for (uint32_t f = 0; f < n_first; f++) {
            const uint32_t p = first[f];
            const unsigned char *pat = pat_blob + pat_off[p];
            const int m = (int)(pat_off[p + 1] - pat_off[p]);
            if (len < m) continue; /* serial.c:193-194 */
            int j = 0;
            for (int64_t i = 0; i < len; i++) { /* serial.c:196-212 */
                while (j > 0 && pat[j] != text[i]) j = pi[p][j - 1];
                if (pat[j] == text[i]) j++;
                if (j == m) {
                    if (n == cap) hits = realloc(hits, (cap *= 2) * sizeof *hits);
                    hits[n].offset = (uint32_t)(i - m + 1);
                    hits[n].pattern = p;
                    n++;
                    j = pi[p][m - 1];
                }
            }
        }
        qsort(hits, n, sizeof *hits, hit_cmp);
        for (size_t h = 0; h < n; h++, total++) {
            if (total >= capacity) continue;
            packet[total] = k;
            offset[total] = hits[h].offset;
            pattern[total] = hits[h].pattern;
        }
    }
    free(hits);
    for (uint32_t p = 0; p < n_pat; p++) free(pi[p]);
    free(pi);
    free(first);
    return total;
}
