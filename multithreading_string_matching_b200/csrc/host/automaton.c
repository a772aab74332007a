/* automaton.c -- host-side table construction for a pattern set (runs once per kmpb_set_patterns).
 *
 * The reference keeps one KMP failure table per pattern (kmp_prefix, serial.c:217-238) and walks
 * every payload once per pattern (serial.c:153-155).  Walking the payload P times cannot come near
 * the HBM roofline, so the union engine reads it once: a 4-byte-deep shift-and prefilter over 5 buckets
 * of patterns (+ a NUL detector) finds the few positions where some pattern can start at all
 * (kmpb_filter6_build), and start-anchored probe tables name the patterns that really do
 * (build_verify_tables).  Counting every occurrence once at its start gives the numbers P independent
 * kmp_matcher calls give (overlapping occurrences are separate occurrences either way).
 *
 * Case-insensitive patterns (KMPB_PAT_NOCASE, kmpb_tables_build_flags) are a matter of these tables alone: such a
 * pattern is stored folded, admits both cases of its letters in the filter and the gate, is entered under every case
 * variant of its probe key, and its records' masks clear bit 5 at its letters.  With every flag zero the tables are
 * word for word those of kmpb_tables_build.
 *
 * For the table tests only (kmpb_tables_build_ex with_dfa): the P KMP automata merged into one DFA over
 * the trie of all pattern prefixes -- state = longest suffix of the text read so far that is a prefix of
 * some pattern; for a single pattern exactly the automaton kmp_matcher steps through (j, with the drop
 * to prefix[j-1] on mismatch or after a hit, serial.c:203-211).  tests/c/test_tables.c checks the filter
 * and the probe tables against it and against a naive counter.
 */
#include <stdlib.h>
#include <string.h>

#include "kmpb_internal.h"

#define N_BUCKET 5        /* pattern buckets; the sixth bit of every field belongs to the NUL detector */
#define FILTER_DEPTH 4
#define TEXT_ALPHABET 96.0 /* cost model only: distinct byte values expected in payload text */
#define DP_LIMIT 1024      /* above this many distinct patterns the bucket split is not optimised */

/* ---- distinct patterns ------------------------------------------------------------------------ */

typedef struct {
    const uint8_t *p; /* folded when nc */
    uint32_t len, index;
    uint32_t nc;      /* KMPB_PAT_NOCASE */
    uint32_t lo, hi;  /* window; {0, KMPB_WINDOW_ANY} = none */
} pat_ref;

static int windowed(const pat_ref *r) { return r->hi != KMPB_WINDOW_ANY; }

/* ASCII case folding (kmpb200.h): A-Z to a-z, every other byte as it is */
static uint8_t fold(uint8_t c) { return c >= 'A' && c <= 'Z' ? (uint8_t)(c + 32) : c; }
/* a byte of a folded nocase pattern that matches two text bytes: a lower-case letter (the other is c ^ 0x20) */
static int folds(uint32_t nc, uint8_t c) { return nc && c >= 'a' && c <= 'z'; }

/* content, then flag */
static int cmp_bytes_flag(const pat_ref *x, const pat_ref *y)
{
    uint32_t n = x->len < y->len ? x->len : y->len;
    int c = memcmp(x->p, y->p, n);
    if (c) return c;
    if (x->len != y->len) return x->len < y->len ? -1 : 1;
    if (x->nc != y->nc) return x->nc < y->nc ? -1 : 1;
    return 0;
}

/* distinct patterns are equal (bytes, flag); the order is content, then flag, then file order */
static int cmp_content(const void *a, const void *b)
{
    const pat_ref *x = a, *y = b;
    const int c = cmp_bytes_flag(x, y);
    if (c) return c;
    return x->index < y->index ? -1 : (x->index > y->index);
}

/* the order of the distinct ids: the patterns without a window first, in content order (so they are numbered as in a
 * set without windows), then the windowed ones by content, flag and window -- so the windowed patterns of one byte
 * and flag have consecutive ids, and the one-byte table of their probe tables, which holds the last of them, leads
 * the window kernel to all of them */
static int cmp_distinct(const void *a, const void *b)
{
    const pat_ref *x = a, *y = b;
    if (windowed(x) != windowed(y)) return windowed(x) - windowed(y);
    const int c = cmp_bytes_flag(x, y);
    if (c) return c;
    if (x->lo != y->lo) return x->lo < y->lo ? -1 : 1;
    if (x->hi != y->hi) return x->hi < y->hi ? -1 : 1;
    return x->index < y->index ? -1 : (x->index > y->index);
}

/* order used for bucketing: by min(len, depth) first so short patterns (which leave the deeper
 * filter stages open) share buckets, then by content so common prefixes sit together */
static int cmp_bucket(const void *a, const void *b)
{
    const pat_ref *x = a, *y = b;
    uint32_t kx = x->len < FILTER_DEPTH ? x->len : FILTER_DEPTH, ky = y->len < FILTER_DEPTH ? y->len : FILTER_DEPTH;
    if (kx != ky) return kx < ky ? -1 : 1;
    return cmp_content(a, b);
}

/* ---- prefilter -------------------------------------------------------------------------------- */

typedef struct {
    uint64_t set[FILTER_DEPTH][4]; /* byte values allowed at each depth */
    int open[FILTER_DEPTH];        /* some pattern is shorter than depth+1: every byte passes */
} bucket_sets;

static void sets_add(bucket_sets *s, const pat_ref *r)
{
    for (uint32_t d = 0; d < FILTER_DEPTH; d++) {
        if (d < r->len) {
            s->set[d][r->p[d] >> 6] |= 1ull << (r->p[d] & 63);
            if (folds(r->nc, r->p[d])) s->set[d][(r->p[d] ^ 0x20) >> 6] |= 1ull << ((r->p[d] ^ 0x20) & 63);
        } else s->open[d] = 1;
    }
}

static double sets_cost(const bucket_sets *s)
{
    double c = 1.0;
    for (uint32_t d = 0; d < FILTER_DEPTH; d++) {
        if (s->open[d]) continue;
        int n = 0;
        for (int w = 0; w < 4; w++) n += __builtin_popcountll(s->set[d][w]);
        double f = n / TEXT_ALPHABET;
        c *= f > 1.0 ? 1.0 : f;
    }
    return c;
}

/* Split the bucket-ordered patterns into <= n_bucket (<= N_BUCKET) contiguous runs minimising the summed
 * per-byte candidate probability.  cut[b]..cut[b+1] is bucket b. */
static double split_buckets(const pat_ref *sorted, uint32_t n, uint32_t *cut, uint32_t n_bucket)
{
    uint32_t nb = n < n_bucket ? n : n_bucket;
    for (uint32_t b = 0; b <= n_bucket; b++) cut[b] = n;
    cut[0] = 0;
    if (n == 0) return 0.0;
    if (n > DP_LIMIT) {
        double total = 0;
        for (uint32_t b = 0; b < nb; b++) {
            cut[b] = (uint32_t)((uint64_t)n * b / nb);
            uint32_t hi = (uint32_t)((uint64_t)n * (b + 1) / nb);
            bucket_sets s;
            memset(&s, 0, sizeof s);
            for (uint32_t i = cut[b]; i < hi; i++) sets_add(&s, &sorted[i]);
            total += sets_cost(&s);
        }
        return total;
    }
    /* cost[i*(n+1)+j] = cost of one bucket holding sorted[i..j) */
    double *cost = malloc((size_t)(n + 1) * (n + 1) * sizeof *cost);
    double *best = malloc((size_t)(nb + 1) * (n + 1) * sizeof *best);
    uint32_t *from = malloc((size_t)(nb + 1) * (n + 1) * sizeof *from);
    for (uint32_t i = 0; i < n; i++) {
        bucket_sets s;
        memset(&s, 0, sizeof s);
        for (uint32_t j = i + 1; j <= n; j++) {
            sets_add(&s, &sorted[j - 1]);
            cost[(size_t)i * (n + 1) + j] = sets_cost(&s);
        }
    }
    for (uint32_t j = 0; j <= n; j++) best[j] = j == 0 ? 0.0 : 1e300;
    for (uint32_t k = 1; k <= nb; k++) {
        double *cur = best + (size_t)k * (n + 1), *prev = best + (size_t)(k - 1) * (n + 1);
        for (uint32_t j = 0; j <= n; j++) {
            cur[j] = 1e300;
            from[(size_t)k * (n + 1) + j] = 0;
            for (uint32_t i = k - 1; i < j; i++) {
                if (prev[i] >= 1e300) continue;
                double c = prev[i] + cost[(size_t)i * (n + 1) + j];
                if (c < cur[j]) {
                    cur[j] = c;
                    from[(size_t)k * (n + 1) + j] = i;
                }
            }
        }
    }
    double total = best[(size_t)nb * (n + 1) + n];
    uint32_t j = n;
    for (uint32_t k = nb; k >= 1; k--) {
        uint32_t i = from[(size_t)k * (n + 1) + j];
        cut[k - 1] = i;
        j = i;
    }
    free(cost);
    free(best);
    free(from);
    return total;
}

/* Buckets as multisets, so that patterns can be moved in and out: per depth, how many members have each
 * byte value there, how many distinct values that makes, and how many members are too short to have one. */
typedef struct {
    uint16_t count[FILTER_DEPTH][256];
    uint32_t distinct[FILTER_DEPTH], open[FILTER_DEPTH], members;
} bucket_bag;

static void bag_change(bucket_bag *g, const pat_ref *r, int add)
{
    for (uint32_t d = 0; d < FILTER_DEPTH; d++) {
        if (d >= r->len) { g->open[d] += add ? 1 : -1; continue; }
        for (int v = 0; v <= folds(r->nc, r->p[d]); v++) { /* a nocase letter: both cases */
            uint16_t *c = &g->count[d][r->p[d] ^ (v ? 0x20 : 0)];
            if (add) { if ((*c)++ == 0) g->distinct[d]++; }
            else if (--(*c) == 0) g->distinct[d]--;
        }
    }
    g->members += add ? 1 : -1;
}

static double bag_cost(const bucket_bag *g)
{
    if (g->members == 0) return 0.0;
    double c = 1.0;
    for (uint32_t d = 0; d < FILTER_DEPTH; d++) {
        if (g->open[d]) continue;
        double f = g->distinct[d] / TEXT_ALPHABET;
        c *= f > 1.0 ? 1.0 : f;
    }
    return c;
}

#define REFINE_LIMIT 512 /* above this many distinct patterns the contiguous split is kept as it is */

/* Hill climbing from the contiguous split: move single patterns, then swap pairs, while the summed
 * candidate probability drops.  bucket[i] = bucket of sorted[i]. */
static double refine_buckets(const pat_ref *sorted, uint32_t n, uint8_t *bucket, uint32_t n_bucket)
{
    bucket_bag *bag = calloc(n_bucket, sizeof *bag);
    if (!bag) return -1.0;
    for (uint32_t i = 0; i < n; i++) bag_change(&bag[bucket[i]], &sorted[i], 1);
    for (int sweep = 0, improved = 1; improved && sweep < 64; sweep++) {
        improved = 0;
        for (uint32_t i = 0; i < n; i++) { /* moves */
            const uint32_t a = bucket[i];
            const double ca = bag_cost(&bag[a]);
            bag_change(&bag[a], &sorted[i], 0);
            const double gain_out = ca - bag_cost(&bag[a]);
            double best = -1e-15;
            uint32_t to = a;
            for (uint32_t b = 0; b < n_bucket; b++) {
                if (b == a) continue;
                const double cb = bag_cost(&bag[b]);
                bag_change(&bag[b], &sorted[i], 1);
                const double delta = bag_cost(&bag[b]) - cb - gain_out;
                bag_change(&bag[b], &sorted[i], 0);
                if (delta < best) { best = delta; to = b; }
            }
            bag_change(&bag[to], &sorted[i], 1);
            if (to != a) { bucket[i] = (uint8_t)to; improved = 1; }
        }
        for (uint32_t i = 0; i < n; i++) /* swaps */
            for (uint32_t j = i + 1; j < n; j++) {
                const uint32_t a = bucket[i], b = bucket[j];
                if (a == b) continue;
                const double before = bag_cost(&bag[a]) + bag_cost(&bag[b]);
                bag_change(&bag[a], &sorted[i], 0); bag_change(&bag[b], &sorted[j], 0);
                bag_change(&bag[a], &sorted[j], 1); bag_change(&bag[b], &sorted[i], 1);
                if (bag_cost(&bag[a]) + bag_cost(&bag[b]) < before - 1e-15) {
                    bucket[i] = (uint8_t)b; bucket[j] = (uint8_t)a; improved = 1;
                } else {
                    bag_change(&bag[a], &sorted[j], 0); bag_change(&bag[b], &sorted[i], 0);
                    bag_change(&bag[a], &sorted[i], 1); bag_change(&bag[b], &sorted[j], 1);
                }
            }
    }
    double total = 0;
    for (uint32_t b = 0; b < n_bucket; b++) total += bag_cost(&bag[b]);
    free(bag);
    return total;
}

/* Filter words for n_bucket pattern buckets in fields of field_bits bits: bit (field_bits * d + b) of words[c] is set
 * when some pattern of bucket b has byte c at depth d (or is shorter than d+1 bytes).  uniq[] is reordered.
 * Returns the estimated candidate probability per text byte. */
static double build_filter_words(uint32_t n_uniq, pat_ref *uniq, uint32_t n_bucket, uint32_t field_bits, uint32_t *words)
{
    uint32_t cut[N_BUCKET + 1];
    qsort(uniq, n_uniq, sizeof *uniq, cmp_bucket);
    double estimate = split_buckets(uniq, n_uniq, cut, n_bucket);
    uint8_t *bucket = malloc(n_uniq ? n_uniq : 1);
    memset(words, 0, 256 * sizeof *words);
    if (bucket) {
        for (uint32_t b = 0; b < n_bucket; b++)
            for (uint32_t i = cut[b]; i < cut[b + 1]; i++) bucket[i] = (uint8_t)b;
        if (n_uniq <= REFINE_LIMIT) {
            double refined = refine_buckets(uniq, n_uniq, bucket, n_bucket);
            if (refined >= 0) estimate = refined;
        }
    }
    for (uint32_t b = 0; b < n_bucket; b++) {
        bucket_sets s;
        memset(&s, 0, sizeof s);
        uint32_t members = 0;
        for (uint32_t i = 0; i < n_uniq; i++)
            if (bucket ? bucket[i] == b : (i >= cut[b] && i < cut[b + 1])) { sets_add(&s, &uniq[i]); members++; }
        if (members == 0) continue;
        for (uint32_t c = 0; c < 256; c++)
            for (uint32_t d = 0; d < FILTER_DEPTH; d++)
                if (s.open[d] || (s.set[d][c >> 6] >> (c & 63) & 1)) words[c] |= 1u << (field_bits * d + b);
    }
    free(bucket);
    return estimate;
}

/* The prefilter in the geometry the union kernel uses: five fields of 6 bits -- depths 0..3 and a fifth field that
 * passes everything, so that a report lingers one step -- with 5 pattern buckets (bits 0..4 of a field) and the NUL
 * detector in bit 5 (depth 0 passes on NUL only, depths 1..3 always: it reports three bytes after the NUL, when a
 * pattern starting at the NUL would report).  One update per byte: S = ((S << 6) | 0x3f) & words[c]; bits 18..22
 * report the windows that end at this byte, bit 23 "the byte three back is NUL", bits 24..29 the same for the byte
 * before.  Two bytes per update (what the row loop does):
 *   S = ((S << 12) | 0xfff) & ((words[b0] << 6) | 0x3f) & words[b1]
 * which is the same function (tests/c/test_tables.c checks it), bits 24..29 then being byte b0's reports.
 * The bucket split starts from the optimal contiguous split of the patterns sorted by (min(len, 4), content) and is
 * refined by hill climbing (moves and swaps) on the estimated candidate probability. */
int kmpb_filter6_build(const kmpb_tables *t, uint32_t words[256], double *estimate)
{
    pat_ref *uniq = malloc((t->n_union ? t->n_union : 1) * sizeof *uniq);
    if (!uniq) return kmpb_fail(KMPB_ENOMEM, "out of memory building the prefilter");
    for (uint32_t u = 0; u < t->n_union; u++) {
        uniq[u].p = t->uniq_blob + t->uniq_off[u];
        uniq[u].len = t->uniq_len[u];
        uniq[u].index = u;
        uniq[u].nc = t->uniq_flags ? t->uniq_flags[u] : 0u;
    }
    const double e = build_filter_words(t->n_union, uniq, N_BUCKET, 6, words);
    free(uniq);
    /* the NUL detector: depth 0 passes on NUL only, depths 1..3 always -- it reports three bytes after the NUL, when a
     * pattern starting at the NUL would report, so that a report's "candidate" and "NUL" bits speak of the same byte */
    for (uint32_t c = 0; c < 256; c++) words[c] |= (0x3fu << 24) | (1u << 11) | (1u << 17) | (1u << 23);
    words[0] |= 1u << 5;
    if (estimate) *estimate = e;
    return KMPB_OK;
}

/* ---- union automaton -------------------------------------------------------------------------- */

/* The merged automaton of the distinct patterns with flag nc, over t's byte classes.  For nocase patterns (stored folded)
 * the column of an upper-case letter is copied from its lower-case letter's: the automaton then reads fold(text). */
typedef struct {
    uint32_t n_state;
    uint32_t *next, *trie, *term, *out_head, *out_id;
} ac_automaton;

static void ac_free(ac_automaton *a)
{
    free(a->next); free(a->trie); free(a->term); free(a->out_head); free(a->out_id);
    memset(a, 0, sizeof *a);
}

static int ac_build(const kmpb_tables *t, uint32_t nc, ac_automaton *a)
{
    memset(a, 0, sizeof *a);
    const uint32_t ncl = t->n_class;
    uint64_t max_state = (uint64_t)t->uniq_off[t->n_union] + 1;
    if (max_state * ncl >= (1ull << 31))
        return kmpb_fail(KMPB_ELIMIT, "pattern set too large: %llu trie states x %u byte classes exceeds 2^31 table entries",
                         (unsigned long long)max_state, ncl);
    uint32_t *next = calloc((size_t)max_state * ncl, sizeof *next); /* 0 = no child yet (root is never a child) */
    uint32_t *term = malloc((size_t)max_state * sizeof *term);      /* uniq id ending at the state, or ~0 */
    uint32_t *fail = calloc((size_t)max_state, sizeof *fail);
    uint32_t *queue = malloc((size_t)max_state * sizeof *queue);
    uint32_t *n_out = calloc((size_t)max_state, sizeof *n_out);
    if (!next || !term || !fail || !queue || !n_out) {
        free(next); free(term); free(fail); free(queue); free(n_out);
        return kmpb_fail(KMPB_ENOMEM, "out of memory building the union automaton");
    }
    memset(term, 0xff, (size_t)max_state * sizeof *term);

    /* trie of all pattern prefixes */
    uint32_t n_state = 1;
    for (uint32_t u = 0; u < t->n_union; u++) {
        if ((t->uniq_flags ? t->uniq_flags[u] : 0u) != nc) continue;
        uint32_t s = 0;
        for (uint32_t i = t->uniq_off[u]; i < t->uniq_off[u + 1]; i++) {
            uint32_t cls = t->byte_class[t->uniq_blob[i]];
            if (next[(size_t)s * ncl + cls] == 0) next[(size_t)s * ncl + cls] = n_state++;
            s = next[(size_t)s * ncl + cls];
        }
        term[s] = u;
    }
    /* nocase: an upper-case letter goes where its lower-case letter goes */
    const uint8_t *bc = t->byte_class;
#define AC_FOLD_COLUMNS(tab)                                                                                  \
    if (nc)                                                                                                   \
        for (uint32_t s_ = 0; s_ < n_state; s_++)                                                             \
            for (int c_ = 'A'; c_ <= 'Z'; c_++)                                                               \
                if (bc[c_] != bc[c_ + 32]) (tab)[(size_t)s_ * ncl + bc[c_]] = (tab)[(size_t)s_ * ncl + bc[c_ + 32]];

    /* the bare trie (goto function only, 0 = no edge), for the start-anchored walk of the table tests: bit 31 of an
     * edge says a pattern ends at the child */
    uint32_t *trie = malloc((size_t)n_state * ncl * sizeof *trie);
    if (!trie) {
        free(next); free(term); free(fail); free(queue); free(n_out);
        return kmpb_fail(KMPB_ENOMEM, "out of memory building the trie");
    }
    for (size_t e = 0; e < (size_t)n_state * ncl; e++)
        trie[e] = next[e] ? (next[e] | (term[next[e]] != 0xffffffffu ? 0x80000000u : 0u)) : 0u;
    AC_FOLD_COLUMNS(trie);

    /* breadth-first: failure link of a child = where the parent's failure state goes on the same
     * byte (the KMP "while j>0 && p[j]!=c: j=prefix[j-1]" loop, resolved once per (state, byte));
     * missing edges are filled with the failure state's edge, turning the trie into a full DFA */
    uint32_t head = 0, tail = 0;
    for (uint32_t cls = 0; cls < ncl; cls++)
        if (next[cls]) queue[tail++] = next[cls]; /* depth-1 states fail to the root */
    while (head < tail) {
        uint32_t s = queue[head++];
        n_out[s] = (term[s] != 0xffffffffu) + n_out[fail[s]];
        for (uint32_t cls = 0; cls < ncl; cls++) {
            uint32_t child = next[(size_t)s * ncl + cls], via = next[(size_t)fail[s] * ncl + cls];
            if (child) {
                fail[child] = via;
                queue[tail++] = child;
            } else {
                next[(size_t)s * ncl + cls] = via;
            }
        }
    }
    AC_FOLD_COLUMNS(next);
#undef AC_FOLD_COLUMNS

    /* outputs: own pattern first (the longest), then the failure chain's */
    uint32_t *out_head = malloc(((size_t)n_state + 1) * sizeof *out_head);
    uint64_t total_out = 0;
    for (uint32_t s = 0; s < n_state; s++) total_out += n_out[s];
    uint32_t *out_id = malloc((size_t)(total_out ? total_out : 1) * sizeof *out_id);
    if (!out_head || !out_id || total_out >= (1ull << 32)) {
        free(next); free(term); free(fail); free(queue); free(n_out); free(out_head); free(out_id); free(trie);
        return kmpb_fail(KMPB_ENOMEM, "out of memory building the output lists");
    }
    uint32_t at = 0;
    for (uint32_t s = 0; s < n_state; s++) {
        out_head[s] = at;
        for (uint32_t v = s; v != 0; v = fail[v])
            if (term[v] != 0xffffffffu) out_id[at++] = term[v];
    }
    out_head[n_state] = at;

    /* "the target state reports something" flag in bit 31 */
    for (size_t e = 0; e < (size_t)n_state * ncl; e++) {
        uint32_t target = next[e];
        next[e] = target | (n_out[target] ? 0x80000000u : 0u);
    }
    uint32_t *shrunk = realloc(next, (size_t)n_state * ncl * sizeof *next);
    a->next = shrunk ? shrunk : next;
    a->n_state = n_state;
    a->out_head = out_head;
    a->out_id = out_id;
    a->trie = trie;
    uint32_t *term_shrunk = realloc(term, (size_t)n_state * sizeof *term);
    a->term = term_shrunk ? term_shrunk : term;
    free(fail); free(queue); free(n_out);
    return KMPB_OK;
}

/* A set of case-sensitive and nocase patterns: the product of the two automata (a state is the pair of their states,
 * its outputs both lists).  Only the pairs reachable from the roots are kept.  There is no bare trie for such a set. */
static int ac_product(const kmpb_tables *t, const ac_automaton *x, const ac_automaton *y, kmpb_tables *out)
{
    const uint32_t ncl = t->n_class;
    const uint64_t pairs = (uint64_t)x->n_state * y->n_state;
    if (pairs >= (1ull << 28)) return kmpb_fail(KMPB_ELIMIT, "mixed pattern set too large for the merged automaton");
    uint32_t *id = calloc(pairs, sizeof *id); /* 1 + state of a pair, 0 = not reached yet */
    uint32_t cap = 1024, n = 1;
    uint32_t *px = malloc(cap * sizeof *px), *py = malloc(cap * sizeof *py);
    uint32_t *next = malloc((size_t)cap * ncl * sizeof *next);
    if (!id || !px || !py || !next) { free(id); free(px); free(py); free(next); return kmpb_fail(KMPB_ENOMEM, "out of memory"); }
    px[0] = 0; py[0] = 0; id[0] = 1;
    for (uint32_t s = 0; s < n; s++)
        for (uint32_t cls = 0; cls < ncl; cls++) {
            const uint32_t a = x->next[(size_t)px[s] * ncl + cls] & 0x7fffffffu, b = y->next[(size_t)py[s] * ncl + cls] & 0x7fffffffu;
            uint32_t *slot = &id[(uint64_t)a * y->n_state + b];
            if (*slot == 0) {
                if (n == cap) {
                    cap *= 2;
                    uint32_t *nx = realloc(px, cap * sizeof *px), *ny = realloc(py, cap * sizeof *py);
                    uint32_t *nn = realloc(next, (size_t)cap * ncl * sizeof *next);
                    if (nx) px = nx;
                    if (ny) py = ny;
                    if (nn) next = nn;
                    if (!nx || !ny || !nn) { free(id); free(px); free(py); free(next); return kmpb_fail(KMPB_ENOMEM, "out of memory"); }
                }
                px[n] = a; py[n] = b;
                *slot = ++n;
            }
            next[(size_t)s * ncl + cls] = *slot - 1;
        }
    uint32_t *out_head = malloc(((size_t)n + 1) * sizeof *out_head);
    uint64_t total = 0;
    for (uint32_t s = 0; s < n; s++)
        total += (x->out_head[px[s] + 1] - x->out_head[px[s]]) + (y->out_head[py[s] + 1] - y->out_head[py[s]]);
    uint32_t *out_id = malloc((size_t)(total ? total : 1) * sizeof *out_id);
    if (!out_head || !out_id) {
        free(id); free(px); free(py); free(next); free(out_head); free(out_id);
        return kmpb_fail(KMPB_ENOMEM, "out of memory");
    }
    uint32_t at = 0;
    for (uint32_t s = 0; s < n; s++) {
        out_head[s] = at;
        for (uint32_t o = x->out_head[px[s]]; o < x->out_head[px[s] + 1]; o++) out_id[at++] = x->out_id[o];
        for (uint32_t o = y->out_head[py[s]]; o < y->out_head[py[s] + 1]; o++) out_id[at++] = y->out_id[o];
    }
    out_head[n] = at;
    for (size_t e = 0; e < (size_t)n * ncl; e++)
        next[e] |= out_head[next[e] + 1] > out_head[next[e]] ? 0x80000000u : 0u;
    free(id); free(px); free(py);
    out->next = next;
    out->n_state = n;
    out->out_head = out_head;
    out->out_id = out_id;
    return KMPB_OK;
}

static int build_dfa(kmpb_tables *t)
{
    /* byte classes: every byte a pattern can match has its own (both cases of a nocase pattern's letters) */
    int used[256] = {0};
    uint32_t has[2] = {0, 0};
    for (uint32_t u = 0; u < t->n_union; u++) {
        const uint32_t nc = t->uniq_flags ? t->uniq_flags[u] : 0u;
        has[nc] = 1;
        for (uint32_t i = t->uniq_off[u]; i < t->uniq_off[u + 1]; i++) {
            used[t->uniq_blob[i]] = 1;
            if (folds(nc, t->uniq_blob[i])) used[t->uniq_blob[i] ^ 0x20] = 1;
        }
    }
    t->n_class = 1;
    for (int c = 0; c < 256; c++) t->byte_class[c] = used[c] ? (uint8_t)t->n_class++ : 0;
    if (t->n_class > 256) { /* all 256 byte values used: cannot happen (no NUL), but keep u8 safe */
        return kmpb_fail(KMPB_ELIMIT, "pattern set uses every byte value");
    }
    ac_automaton a[2];
    int rc = ac_build(t, has[1] && !has[0] ? 1u : 0u, &a[0]);
    if (rc) return rc;
    if (!(has[0] && has[1])) { /* one kind of pattern: its automaton */
        t->next = a[0].next; t->n_state = a[0].n_state; t->out_head = a[0].out_head; t->out_id = a[0].out_id;
        t->trie = a[0].trie; t->state_term = a[0].term;
        return KMPB_OK;
    }
    rc = ac_build(t, 1u, &a[1]);
    if (rc == KMPB_OK) rc = ac_product(t, &a[0], &a[1], t);
    ac_free(&a[0]);
    ac_free(&a[1]);
    return rc;
}

/* ---- start-anchored verification tables ---------------------------------------------------------- */

#define VT_HEADER 8

/* slot of a text position's first bytes (little-endian, masked to the key length by the caller) in a table of
 * 1 << (32 - shift) slots */
uint32_t kmpb_vtab_slot(uint32_t key, uint32_t shift) { return (key * 0x9e3779b1u) >> shift; }

static uint32_t word_of(const uint8_t *p, uint32_t len, uint32_t from)
{
    uint32_t k = 0;
    for (uint32_t i = from; i < from + 4 && i < len; i++) k |= (uint32_t)p[i] << (8 * (i - from));
    return k;
}
static uint32_t mask_of(const uint8_t *p, uint32_t len, uint32_t nc, uint32_t from)
{
    uint32_t k = 0;
    for (uint32_t i = from; i < from + 4 && i < len; i++) k |= (folds(nc, p[i]) ? 0xdfu : 0xffu) << (8 * (i - from));
    return k;
}

/* key of a pattern in its probe table: A = the two-byte patterns (their two bytes), B = three and more bytes
 * (the first three) */
static uint32_t vt_key(const uint8_t *p, uint32_t len) { return word_of(p, len < 3 ? len : 3, 0); }

/* The keys a text position that matches the pattern can have: the pattern's own, and for a nocase pattern every case
 * variant of the letters among its key bytes (at most 8).  Returns how many; keys[0] is the pattern's own. */
static uint32_t vt_keys(const uint8_t *p, uint32_t len, uint32_t nc, uint32_t keys[8])
{
    const uint32_t kl = len < 3 ? len : 3;
    uint32_t n = 1;
    keys[0] = vt_key(p, len);
    for (uint32_t i = 0; i < kl; i++)
        if (folds(nc, p[i]))
            for (uint32_t j = 0, m = n; j < m; j++) keys[n++] = keys[j] ^ (0x20u << (8 * i));
    return n;
}

/* The distinct probe-table slots of those keys (two case variants can hash to one slot: the pattern's record goes in
 * once).  Returns how many. */
static uint32_t vt_slots(const uint8_t *p, uint32_t len, uint32_t nc, uint32_t shift, uint32_t slots[8])
{
    uint32_t keys[8], n = 0;
    const uint32_t nk = vt_keys(p, len, nc, keys);
    for (uint32_t k = 0; k < nk; k++) {
        const uint32_t s = kmpb_vtab_slot(keys[k], shift);
        uint32_t j = 0;
        while (j < n && slots[j] != s) j++;
        if (j == n) slots[n++] = s;
    }
    return n;
}

/* The probe tables of distinct ids [u0, u0 + n), n_nocase of them nocase, into *out (*out_words words): vtab for
 * the patterns without a window, wvtab for the windowed ones. */
static int build_verify_tables(const kmpb_tables *t, uint32_t u0, uint32_t n, uint32_t n_nocase, uint32_t **out,
                               uint32_t *out_words)
{
    /* Two probe tables, one slot per hash value of the key, at least four slots per key: most slots are empty and
     * most occupied slots hold the patterns of a single key.  Keying the longer patterns by three bytes instead of two
     * (round 1) cuts the longest chain of strings.txt from 6 records ("se..") to 3 ("htt", "por") -- a warp walks as
     * many records as its longest chain.  A nocase pattern is entered under every case variant of its key. */
    uint32_t n_a = 0, n_b = 0, n1 = 0, blob_words = 0, mask_words = 0, keys[8];
    for (uint32_t u = u0; u < u0 + n; u++) {
        const uint8_t *p = t->uniq_blob + t->uniq_off[u];
        const uint32_t len = t->uniq_len[u], nc = t->uniq_flags[u];
        if (len >= 3) n_b += vt_keys(p, len, nc, keys); else if (len == 2) n_a += vt_keys(p, len, nc, keys); else n1++;
        blob_words += (len + 3) / 4;
        if (nc && len > 8) mask_words += (len + 3) / 4;
    }
    uint32_t log_a = 4, log_b = 6;
    while (log_a < 16 && (1u << log_a) < 4 * n_a) log_a++;
    while (log_b < 20 && (1u << log_b) < 4 * n_b) log_b++;
    const uint32_t slots_a = n_a ? 1u << log_a : 0, slots_b = n_b ? 1u << log_b : 0;
    /* records: one per pattern and distinct slot */
    uint32_t n_rec = 0, sl[8];
    for (uint32_t u = u0; u < u0 + n; u++) {
        const uint32_t len = t->uniq_len[u];
        if (len >= 2) n_rec += vt_slots(t->uniq_blob + t->uniq_off[u], len, t->uniq_flags[u], len >= 3 ? 32 - log_b : 32 - log_a, sl);
    }
    uint32_t at = VT_HEADER;
    const uint32_t slot_a_off = n_a ? at : 0;
    at += 2 * slots_a;
    const uint32_t slot_b_off = n_b ? at : 0;
    at += 2 * slots_b;
    /* the one-byte table: 256 words of case-sensitive ids, then -- in a set with a nocase pattern -- 256 of nocase ids,
     * so that `A` and nocase `a` can both claim byte `A` */
    const uint32_t one_off = n1 ? at : 0;
    if (n1) at += n_nocase ? 512 : 256;
    at = (at + 3u) & ~3u; /* records are read 16 bytes at a time */
    const uint32_t rec_off = at;
    at += 8 * n_rec;
    const uint32_t blob_off = at;
    at += blob_words;
    const uint32_t mask_off = at; /* the masks of the nocase patterns of more than 8 bytes, laid out like their words */
    at += mask_words;
    uint32_t *v = calloc(at ? at : 1, sizeof *v);
    uint32_t *fill = calloc((size_t)slots_a + slots_b + 1, sizeof *fill);
    if (!v || !fill) { free(v); free(fill); return kmpb_fail(KMPB_ENOMEM, "out of memory building the verification tables"); }
    v[0] = at; v[1] = slot_a_off; v[2] = 32 - log_a; v[3] = slot_b_off; v[4] = 32 - log_b; v[5] = one_off;
    v[6] = rec_off; v[7] = blob_off;
    for (uint32_t i = 0; n1 && i < (n_nocase ? 512u : 256u); i++) v[one_off + i] = 0xffffffffu;
    /* chain lengths, then chain starts (records of one slot are contiguous; table A's records come first) */
    for (uint32_t u = u0; u < u0 + n; u++) {
        const uint8_t *p = t->uniq_blob + t->uniq_off[u];
        const uint32_t len = t->uniq_len[u];
        if (len < 2) continue;
        const uint32_t ns = vt_slots(p, len, t->uniq_flags[u], len >= 3 ? 32 - log_b : 32 - log_a, sl);
        for (uint32_t k = 0; k < ns; k++) v[(len >= 3 ? slot_b_off : slot_a_off) + 2 * sl[k] + 1]++;
    }
    uint32_t first = 0;
    for (uint32_t s = 0; s < slots_a; s++) { v[slot_a_off + 2 * s] = first; first += v[slot_a_off + 2 * s + 1]; }
    for (uint32_t s = 0; s < slots_b; s++) { v[slot_b_off + 2 * s] = first; first += v[slot_b_off + 2 * s + 1]; }
    uint32_t bw = 0, mw = 0;
    for (uint32_t u = u0; u < u0 + n; u++) {
        const uint8_t *p = t->uniq_blob + t->uniq_off[u];
        const uint32_t len = t->uniq_len[u], nc = t->uniq_flags[u];
        memcpy((uint8_t *)(v + blob_off + bw), p, len); /* rest of the last word stays zero */
        /* a nocase pattern's masks clear bit 5 at its letters: the masked compare then accepts exactly the case
         * variants (the only byte that differs from a letter in bit 5 alone is the same letter in the other case) */
        const uint32_t tail = nc && len > 8 ? mask_off + mw : 0;
        for (uint32_t w = 0; tail && w < (len + 3) / 4; w++) v[tail + w] = mask_of(p, len, nc, 4 * w);
        if (len >= 2) {
            const uint32_t so = len >= 3 ? slot_b_off : slot_a_off, fo = len >= 3 ? slots_a : 0;
            const uint32_t ns = vt_slots(p, len, nc, len >= 3 ? 32 - log_b : 32 - log_a, sl);
            for (uint32_t k = 0; k < ns; k++) {
                uint32_t *rec = v + rec_off + 8 * (v[so + 2 * sl[k]] + fill[fo + sl[k]]++);
                rec[0] = word_of(p, len, 0); rec[1] = mask_of(p, len, nc, 0);
                rec[2] = word_of(p, len, 4); rec[3] = mask_of(p, len, nc, 4);
                rec[4] = len; rec[5] = u; rec[6] = bw; rec[7] = tail;
            }
        } else if (folds(nc, p[0])) {
            v[one_off + 256 + p[0]] = v[one_off + 256 + (p[0] ^ 0x20)] = u;
        } else {
            v[one_off + (nc ? 256 : 0) + p[0]] = u;
        }
        bw += (len + 3) / 4;
        if (tail) mw += (len + 3) / 4;
    }
    free(fill);
    *out = v;
    *out_words = at;
    return KMPB_OK;
}

/* The window kernel's tables: the windowed patterns' probe tables, their windows' extremes and reach, and the bytes
 * they can start with (both cases of a nocase pattern's letter). */
static int build_window_tables(kmpb_tables *t)
{
    const uint32_t nw = t->n_uniq - t->n_union;
    if (nw == 0) return KMPB_OK;
    t->win_lo_min = KMPB_WINDOW_MAX;
    for (uint32_t w = 0; w < nw; w++) {
        const uint32_t u = t->n_union + w, len = t->uniq_len[u];
        const uint8_t c = t->uniq_blob[t->uniq_off[u]];
        if (t->uniq_lo[w] < t->win_lo_min) t->win_lo_min = t->uniq_lo[w];
        if (t->uniq_hi[w] > t->win_hi_max) t->win_hi_max = t->uniq_hi[w];
        if (t->uniq_hi[w] + len > t->win_reach) t->win_reach = t->uniq_hi[w] + len;
        t->win_nocase += t->uniq_flags[u];
        t->win_first[c >> 5] |= 1u << (c & 31);
        if (folds(t->uniq_flags[u], c)) t->win_first[(c ^ 0x20) >> 5] |= 1u << ((c ^ 0x20) & 31);
    }
    return build_verify_tables(t, t->n_union, nw, t->win_nocase, &t->wvtab, &t->wvtab_words);
}

/* ---- prefix gate ------------------------------------------------------------------------------ */

#define GATE_MIN_WORDS 32u
#define GATE_MAX_WORDS 1024u /* 4 KB: what is left of the block's shared memory next to the probe tables of a small set */
#define GATE_WORDS_PER_KEY 16u

uint32_t kmpb_gate_slot(uint32_t x, uint32_t shift) { return (x * KMPB_GATE_MUL) >> shift; }

/* The resolve step's test of a start position before it becomes a candidate (union_kernel.cu, phase 1): the position's
 * first two bytes pick a word, its third byte a bit.  Every pattern sets the bit of its own start, so the gate lets
 * every true start through; what it rejects are the filter's false starts (the short patterns' buckets admit byte
 * combinations no pattern has).  One word per 16 distinct two-byte keys or more (a one-byte pattern is 256 keys); when
 * more than an eighth of the bits end up set, the gate would reject too little and is not built. */
static int build_gate(kmpb_tables *t)
{
    uint32_t keys = 0, last = 0xffffffffu; /* distinct patterns are in content order: equal first two bytes are adjacent */
    for (uint32_t u = 0; u < t->n_union; u++) {
        const uint8_t *p = t->uniq_blob + t->uniq_off[u];
        const uint32_t nc = t->uniq_flags[u];
        if (t->uniq_len[u] == 1) { keys += 256u << folds(nc, p[0]); continue; }
        if (nc) { keys += 1u << (folds(nc, p[0]) + folds(nc, p[1])); continue; } /* its case variants */
        const uint32_t k = p[0] | (uint32_t)p[1] << 8;
        keys += k != last;
        last = k;
    }
    uint32_t log_w = 5;
    while ((1u << log_w) < GATE_MAX_WORDS && (1u << log_w) < GATE_WORDS_PER_KEY * keys) log_w++;
    const uint32_t words = 1u << log_w, shift = 32 - log_w;
    uint32_t *g = calloc(words, sizeof *g);
    if (!g) return kmpb_fail(KMPB_ENOMEM, "out of memory building the prefix gate");
    for (uint32_t u = 0; u < t->n_union; u++) {
        const uint8_t *p = t->uniq_blob + t->uniq_off[u];
        const uint32_t len = t->uniq_len[u], nc = t->uniq_flags[u];
        /* a nocase pattern sets the bits of every case variant of its first two bytes; the bit, third byte & 31, is the
         * same for both cases of a letter */
        for (uint32_t v0 = 0; v0 <= (uint32_t)folds(nc, p[0]); v0++) {
            const uint32_t b0 = p[0] ^ (v0 << 5);
            if (len == 1) {
                for (uint32_t c = 0; c < 256; c++) g[kmpb_gate_slot(b0 | c << 8, shift)] = 0xffffffffu;
                continue;
            }
            for (uint32_t v1 = 0; v1 <= (uint32_t)folds(nc, p[1]); v1++)
                g[kmpb_gate_slot(b0 | (uint32_t)(p[1] ^ (v1 << 5)) << 8, shift)] |= len == 2 ? 0xffffffffu : 0x80000000u >> (p[2] & 31);
        }
    }
    uint64_t set = 0;
    for (uint32_t i = 0; i < words; i++) set += (uint64_t)__builtin_popcount(g[i]);
    if (t->n_union == 0 || 8 * set > 32ull * words) {
        free(g);
        return KMPB_OK;
    }
    t->gate = g;
    t->gate_words = words;
    t->gate_shift = shift;
    return KMPB_OK;
}

/* ---- entry points ----------------------------------------------------------------------------- */

int kmpb_tables_build(kmpb_tables *t, const uint8_t *blob, const uint32_t *pat_off, uint32_t n_pat)
{
    return kmpb_tables_build_flags(t, blob, pat_off, n_pat, NULL, 0);
}

int kmpb_tables_build_ex(kmpb_tables *t, const uint8_t *blob, const uint32_t *pat_off, uint32_t n_pat, int with_dfa)
{
    return kmpb_tables_build_flags(t, blob, pat_off, n_pat, NULL, with_dfa);
}

int kmpb_tables_build_flags(kmpb_tables *t, const uint8_t *blob, const uint32_t *pat_off, uint32_t n_pat,
                            const uint8_t *flags, int with_dfa)
{
    return kmpb_tables_build_win(t, blob, pat_off, n_pat, flags, NULL, with_dfa);
}

/* with_dfa != 0 also builds the merged automaton of all patterns without a window (next / trie / out_*): the reference
 * the table tests check the filter and the verification tables against.  The device never sees it, so the library does
 * not build it.  flags[n_pat] (NULL: all zero) holds each pattern's KMPB_PAT_* bits, win[n_pat] (NULL: none) its
 * window. */
int kmpb_tables_build_win(kmpb_tables *t, const uint8_t *blob, const uint32_t *pat_off, uint32_t n_pat,
                          const uint8_t *flags, const kmpb_window *win, int with_dfa)
{
    memset(t, 0, sizeof *t);
    if (n_pat && (blob == NULL || pat_off == NULL)) return kmpb_fail(KMPB_EINVAL, "kmpb_set_patterns: NULL pattern data");
    t->n_pat = n_pat;
    pat_ref *refs = malloc(((size_t)n_pat + 1) * sizeof *refs);
    t->pat_to_uniq = malloc(((size_t)n_pat + 1) * sizeof *t->pat_to_uniq);
    if (!refs || !t->pat_to_uniq) { free(refs); kmpb_tables_free(t); return kmpb_fail(KMPB_ENOMEM, "out of memory"); }
    uint64_t blob_len = 0;
    for (uint32_t i = 0; i < n_pat; i++) {
        if (pat_off[i + 1] < pat_off[i]) { free(refs); kmpb_tables_free(t); return kmpb_fail(KMPB_EINVAL, "pattern offsets decrease at %u", i); }
        uint32_t len = pat_off[i + 1] - pat_off[i];
        if (len == 0 || len > KMPB_MAX_PATTERN_LEN) {
            free(refs); kmpb_tables_free(t);
            return kmpb_fail(KMPB_EINVAL, "pattern %u has %u bytes; 1..%d allowed (serial.c:64)", i, len, KMPB_MAX_PATTERN_LEN);
        }
        if (memchr(blob + pat_off[i], 0, len)) {
            free(refs); kmpb_tables_free(t);
            return kmpb_fail(KMPB_EINVAL, "pattern %u contains a NUL byte", i);
        }
        if (flags && (flags[i] & ~KMPB_PAT_NOCASE)) {
            free(refs); kmpb_tables_free(t);
            return kmpb_fail(KMPB_EINVAL, "pattern %u has unknown flag bits 0x%02x", i, flags[i] & ~KMPB_PAT_NOCASE);
        }
        refs[i].p = blob + pat_off[i];
        refs[i].len = len;
        refs[i].index = i;
        refs[i].nc = flags ? flags[i] & KMPB_PAT_NOCASE : 0u;
        refs[i].lo = win ? win[i].lo : 0u;
        refs[i].hi = win ? win[i].hi : KMPB_WINDOW_ANY;
        if (refs[i].lo == 0 && refs[i].hi == KMPB_WINDOW_ANY) { /* no window */
        } else if (refs[i].hi == KMPB_WINDOW_ANY) {
            free(refs); kmpb_tables_free(t);
            return kmpb_fail(KMPB_EINVAL, "pattern %u has window [%u, any]: a window open at the top is not supported", i, win[i].lo);
        } else if (refs[i].lo > refs[i].hi || refs[i].hi > KMPB_WINDOW_MAX) {
            free(refs); kmpb_tables_free(t);
            return kmpb_fail(KMPB_EINVAL, "pattern %u has window [%u, %u]; 0 <= lo <= hi <= %u required", i, win[i].lo,
                             win[i].hi, KMPB_WINDOW_MAX);
        }
        blob_len += len;
    }
    /* nocase patterns are matched in their folded form */
    uint8_t *folded = malloc(blob_len ? blob_len : 1);
    if (!folded) { free(refs); kmpb_tables_free(t); return kmpb_fail(KMPB_ENOMEM, "out of memory"); }
    for (uint64_t i = 0, at = 0; i < n_pat; at += refs[i].len, i++) {
        for (uint32_t k = 0; k < refs[i].len; k++) folded[at + k] = refs[i].nc ? fold(refs[i].p[k]) : refs[i].p[k];
        refs[i].p = folded + at;
    }
    /* distinct patterns: those without a window numbered in content order, then the windowed ones */
    qsort(refs, n_pat, sizeof *refs, cmp_distinct);
    t->uniq_off = malloc(((size_t)n_pat + 1) * sizeof *t->uniq_off);
    t->uniq_len = malloc(((size_t)n_pat + 1) * sizeof *t->uniq_len);
    t->uniq_flags = calloc((size_t)n_pat + 1, 1);
    t->uniq_blob = malloc(blob_len ? blob_len : 1);
    pat_ref *uniq = malloc(((size_t)n_pat + 1) * sizeof *uniq);
    t->uniq_lo = malloc(((size_t)n_pat + 1) * sizeof *t->uniq_lo);
    t->uniq_hi = malloc(((size_t)n_pat + 1) * sizeof *t->uniq_hi);
    if (!t->uniq_off || !t->uniq_len || !t->uniq_flags || !t->uniq_blob || !uniq || !t->uniq_lo || !t->uniq_hi) {
        free(refs); free(uniq); free(folded); kmpb_tables_free(t);
        return kmpb_fail(KMPB_ENOMEM, "out of memory");
    }
    uint32_t nu = 0, at = 0;
    t->min_len = n_pat ? KMPB_MAX_PATTERN_LEN : 0;
    for (uint32_t i = 0; i < n_pat; i++) {
        int same = i > 0 && refs[i].len == refs[i - 1].len && refs[i].nc == refs[i - 1].nc &&
                   refs[i].lo == refs[i - 1].lo && refs[i].hi == refs[i - 1].hi &&
                   memcmp(refs[i].p, refs[i - 1].p, refs[i].len) == 0;
        if (!same) {
            t->uniq_off[nu] = at;
            t->uniq_len[nu] = refs[i].len;
            t->uniq_flags[nu] = (uint8_t)refs[i].nc;
            if (windowed(&refs[i])) {
                t->uniq_lo[nu - t->n_union] = refs[i].lo;
                t->uniq_hi[nu - t->n_union] = refs[i].hi;
            } else {
                t->n_nocase += refs[i].nc;
                t->n_union = nu + 1;
            }
            memcpy(t->uniq_blob + at, refs[i].p, refs[i].len);
            uniq[nu].p = t->uniq_blob + at;
            uniq[nu].len = refs[i].len;
            uniq[nu].index = nu;
            uniq[nu].nc = refs[i].nc;
            at += refs[i].len;
            nu++;
            if (refs[i].len > t->max_len) t->max_len = refs[i].len;
            if (refs[i].len < t->min_len) t->min_len = refs[i].len;
        }
        t->pat_to_uniq[refs[i].index] = nu - 1;
    }
    t->uniq_off[nu] = at;
    t->n_uniq = nu;
    free(refs);
    free(folded);

    int rc = with_dfa ? build_dfa(t) : KMPB_OK;
    if (rc == KMPB_OK) rc = build_verify_tables(t, 0, t->n_union, t->n_nocase, &t->vtab, &t->vtab_words);
    if (rc == KMPB_OK) rc = build_window_tables(t);
    if (rc == KMPB_OK) rc = build_gate(t);
    if (rc == KMPB_OK) rc = kmpb_filter6_build(t, t->filter6, &t->filter6_fp_estimate);
    free(uniq);
    if (rc != KMPB_OK) kmpb_tables_free(t);
    return rc;
}

void kmpb_tables_free(kmpb_tables *t)
{
    free(t->pat_to_uniq);
    free(t->uniq_len);
    free(t->uniq_off);
    free(t->uniq_blob);
    free(t->uniq_flags);
    free(t->next);
    free(t->trie);
    free(t->state_term);
    free(t->out_head);
    free(t->out_id);
    free(t->vtab);
    free(t->gate);
    free(t->uniq_lo);
    free(t->uniq_hi);
    free(t->wvtab);
    memset(t, 0, sizeof *t);
}
