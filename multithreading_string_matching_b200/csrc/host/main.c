/* main.c -- kmp_match: the reference's command line on a B200.
 *
 *   kmp_match <file.pcap> <string.txt> [udp|tcp]            serial.c:3,33-51
 *   kmp_match <file.pcap> <string.txt> <n> [tcp|udp]        openmp_data.c:2,35-54; <n> = number of
 *                                                           GPUs (the reference's thread count)
 *   kmp_match -i <file.pcap> <string.txt> [n] [udp|tcp]     every token case-insensitive (ASCII letters,
 *                                                           KMPB_PAT_NOCASE); the report lists each token as
 *                                                           the strings file spells it
 *   kmp_match -w LO:HI <file.pcap> <string.txt> ...         every token counted only where it starts at a
 *                                                           payload offset in [LO, HI] (kmpb_set_patterns_win,
 *                                                           cli_window.h); -i and -w combine, in either order
 *
 * stdout is the reference's, byte for byte (serial.c:163-169): header line, one "pattern: N times!"
 * line per pattern with a non-zero count in file order, then "Elapsed time = %f seconds" -- the
 * interval covers what serial.c's covers (read + extract + match, serial.c:110-111,159-160).
 * Usage text goes to stdout with exit status 1 (serial.c:43,49); an unreadable strings file is
 * perror("error opening file: ") + exit 1 (serial.c:60-63); an unreadable pcap is "error reading pcap
 * file: ..." on stderr + exit 1 (serial.c:92-95).  Throughput figures go to stderr when KMPB_STATS=1.
 *
 * One host thread drives each GPU: it builds the context while the main thread frames the savefile,
 * then streams its share of the packets (split as mpi_dumping.c:149-157 splits them over ranks) through
 * kmpb_count_pcap; the per-pattern count vectors are summed at the end (mpi_dumping.c:202).
 */
#include <errno.h>
#include <pthread.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <sys/time.h>

#include "cli_window.h"
#include "kmpb200.h"

static double now_seconds(void)
{
    struct timeval tv; /* gettimeofday like timer.h:31-35 */
    gettimeofday(&tv, NULL);
    return (double)tv.tv_sec + (double)tv.tv_usec / 1e6;
}

/* What the GPU threads wait for: the savefile index (or the news that it could not be read). */
typedef struct {
    pthread_mutex_t lock;
    pthread_cond_t ready;
    const kmpb_pcap *pc;
    int done, n_gpus;
} ingest_gate;

typedef struct {
    int device; /* CUDA ordinal */
    int rank;   /* which share of the packets */
    const kmpb_patterns *pats;
    const uint8_t *flags; /* per-pattern KMPB_PAT_* flags, NULL = none */
    const kmpb_window *win; /* per-pattern windows, NULL = none */
    ingest_gate *gate;
    uint64_t *counts;
    double start;
    int rc;
    char err[512];
    kmpb_ctx *ctx; /* kept until the report is out: freeing pinned buffers is not part of the answer */
} shard_job;

/* One host thread per GPU: the context and the pattern tables are built while the main thread frames
 * the savefile; then the GPU's share of the packets (mpi_dumping.c:149-157) streams through it. */
static void *run_shard(void *arg)
{
    shard_job *job = arg;
    kmpb_ctx *ctx = NULL;
    job->rc = kmpb_create(&ctx, job->device);
    if (job->rc == 0) job->rc = kmpb_set_patterns_win(ctx, job->pats->blob, job->pats->pat_off, job->pats->n_pat, job->flags, job->win);
    if (job->rc == 0) job->rc = kmpb_reserve_staging(ctx, 0, 0); /* pinned staging, while the main thread frames the savefile */
    if (job->rc != 0) snprintf(job->err, sizeof job->err, "%s", kmpb_last_error());
    if (getenv("KMPB_STATS")) fprintf(stderr, "kmp_match: GPU %d context, pattern tables and staging buffers ready %.3f s after start\n", job->device, now_seconds() - job->start);
    pthread_mutex_lock(&job->gate->lock);
    while (!job->gate->done) pthread_cond_wait(&job->gate->ready, &job->gate->lock);
    const kmpb_pcap *pc = job->gate->pc;
    pthread_mutex_unlock(&job->gate->lock);
    if (job->rc == 0 && pc != NULL) {
        uint64_t first, count;
        kmpb_shard_range(kmpb_pcap_packets(pc), (uint32_t)job->gate->n_gpus, (uint32_t)job->rank, &first, &count);
        job->rc = kmpb_count_pcap(ctx, pc, first, count, job->counts);
        if (job->rc != 0) snprintf(job->err, sizeof job->err, "%s", kmpb_last_error());
    }
    job->ctx = ctx;
    return NULL;
}

int main(int argc, char **argv)
{
    int proto = KMPB_PROTO_UDP, n_gpus = 1, openmp_form = 0;
    const char *prog = "./kmp_match";
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
    if (argc >= 4 && strcmp(argv[3], "udp") != 0 && strcmp(argv[3], "tcp") != 0 && atoi(argv[3]) > 0) openmp_form = 1;
    const char *usage_colon = openmp_form ? "USAGE: %s <file.pcap> <string.txt> gpu_number [tcp/udp]\n"
                                          : "USAGE: %s <file.pcap> <string.txt> [tcp/udp]\n";
    const char *usage_plain = openmp_form ? "USAGE %s <file.pcap> <string.txt> gpu_number [tcp/udp]\n"
                                          : "USAGE %s <file.pcap> <string.txt> [tcp/udp]\n";
    int type_arg = openmp_form ? 4 : 3;
    if (argc < 3 || argc > type_arg + 1) {
        printf(usage_colon, prog);
        return 1;
    }
    if (openmp_form) n_gpus = atoi(argv[3]);
    if (argc == type_arg + 1) {
        if (strcmp(argv[type_arg], "udp") == 0) proto = KMPB_PROTO_UDP;
        else if (strcmp(argv[type_arg], "tcp") == 0) proto = KMPB_PROTO_TCP;
        else {
            printf(usage_plain, prog);
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

    int available = kmpb_device_count();
    if (available <= 0) {
        fprintf(stderr, "error: no B200-class CUDA device available (this program has no CPU path)\n");
        return 1;
    }
    if (n_gpus > available) n_gpus = available;
    uint8_t *flags = nocase ? malloc(pats.n_pat ? pats.n_pat : 1) : NULL;
    if (flags) memset(flags, KMPB_PAT_NOCASE, pats.n_pat);
    kmpb_window *win = window_array(windowed ? &window : NULL, pats.n_pat);
    if (windowed && win == NULL) {
        fprintf(stderr, "error: out of memory\n");
        return 1;
    }

    double start = now_seconds();
    ingest_gate gate;
    pthread_mutex_init(&gate.lock, NULL);
    pthread_cond_init(&gate.ready, NULL);
    gate.pc = NULL;
    gate.done = 0;
    gate.n_gpus = n_gpus;
    uint64_t *counts = calloc(pats.n_pat ? pats.n_pat : 1, sizeof *counts);
    shard_job *jobs = calloc((size_t)n_gpus, sizeof *jobs);
    pthread_t *threads = calloc((size_t)n_gpus, sizeof *threads);
    for (int g = 0; g < n_gpus; g++) {
        jobs[g].device = kmpb_device_ordinal(g); /* the g-th usable GPU, whatever else the box holds */
        jobs[g].rank = g;
        jobs[g].pats = &pats;
        jobs[g].flags = flags;
        jobs[g].win = win;
        jobs[g].gate = &gate;
        jobs[g].start = start;
        jobs[g].counts = calloc(pats.n_pat ? pats.n_pat : 1, sizeof(uint64_t));
        pthread_create(&threads[g], NULL, run_shard, &jobs[g]);
    }
    kmpb_pcap *pc = NULL;
    rc = kmpb_pcap_open(argv[1], proto, &pc);
    if (getenv("KMPB_STATS")) fprintf(stderr, "kmp_match: savefile framed in %.3f s\n", now_seconds() - start);
    char open_err[512] = "";
    if (rc != 0) snprintf(open_err, sizeof open_err, "%s", kmpb_last_error());
    pthread_mutex_lock(&gate.lock);
    gate.pc = pc;
    gate.done = 1;
    pthread_cond_broadcast(&gate.ready);
    pthread_mutex_unlock(&gate.lock);
    for (int g = 0; g < n_gpus; g++) pthread_join(threads[g], NULL);
    if (rc != 0) {
        fprintf(stderr, "error reading pcap file: %s\n", open_err);
        return 1;
    }
    for (int g = 0; g < n_gpus; g++) {
        if (jobs[g].rc != 0) {
            fprintf(stderr, "error: GPU %d: %s\n", g, jobs[g].err);
            return 1;
        }
        for (uint32_t i = 0; i < pats.n_pat; i++) counts[i] += jobs[g].counts[i];
    }
    double finish = now_seconds();

    kmpb_print_report(stdout, &pats, counts);
    printf("Elapsed time = %f seconds\n", finish - start);

    if (getenv("KMPB_STATS")) {
        double s = finish - start;
        fprintf(stderr, "kmp_match: %llu frames, %llu payloads, %llu payload bytes, %u patterns, %d GPU(s): "
                        "%.3f GB/s, %.3f Mpackets/s end to end (file read + pack + H2D + match)\n",
                (unsigned long long)kmpb_pcap_frames(pc), (unsigned long long)kmpb_pcap_packets(pc),
                (unsigned long long)kmpb_pcap_bytes(pc), pats.n_pat, n_gpus,
                (double)kmpb_pcap_bytes(pc) / s / 1e9, (double)kmpb_pcap_packets(pc) / s / 1e6);
    }
    for (int g = 0; g < n_gpus; g++) {
        kmpb_destroy(jobs[g].ctx);
        free(jobs[g].counts);
    }
    free(jobs);
    free(threads);
    free(counts);
    free(flags);
    free(win);
    kmpb_pcap_close(pc);
    kmpb_free_patterns(&pats);
    return 0;
}
