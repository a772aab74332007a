// tables.cu -- pattern-set tables on the device.
//
// The KMP failure tables (kmp_prefix, serial.c:217-238) are built ON THE DEVICE, one thread per
// distinct pattern, and expanded on the device into byte-indexed transition DFAs (one row of 256
// entries per state) for the per-pattern engine.  The union engine's prefilter and start-anchored hash
// tables come from csrc/host/automaton.c and are uploaded here (the merged automaton itself stays on the
// host, where tests/c/test_tables.c checks the tables against it).
#include <stdlib.h>
#include <string.h>

#include "kmpb_device.cuh"

// pi[i] = length of the longest proper border of pattern[0..i]; same recurrence the reference runs
// on the host for every pattern before matching (serial.c:150-152).
__global__ void kmpb_build_prefix_kernel(const uint8_t *__restrict__ blob, const uint32_t *__restrict__ off,
                                         uint32_t n_uniq, int32_t *__restrict__ pi)
{
    uint32_t u = blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= n_uniq) return;
    const uint8_t *p = blob + off[u];
    int32_t *out = pi + off[u];
    int m = (int)(off[u + 1] - off[u]);
    int border = 0;
    out[0] = 0;
    for (int i = 1; i < m; i++) {
        while (border > 0 && p[i] != p[border]) border = out[border - 1];
        if (p[i] == p[border]) border++;
        out[i] = border;
    }
}

// One block per distinct pattern, one thread per byte value: column c of the pattern's DFA.
// Entry = next state (0..m-1) | 0x80 when the transition completes the pattern; after a hit the
// state drops to pi[m-1] exactly as kmp_matcher does (serial.c:203-206), so m states suffice.
// A nocase pattern (flags[u], its bytes folded) reads the folded text: column c is column fold(c).
__global__ void kmpb_expand_dfa_kernel(const uint8_t *__restrict__ blob, const uint32_t *__restrict__ off,
                                       const uint8_t *__restrict__ flags, const int32_t *__restrict__ pi,
                                       uint8_t *__restrict__ dfa)
{
    uint32_t u = blockIdx.x;
    uint32_t c = threadIdx.x;
    const uint32_t fc = (flags[u] & KMPB_PAT_NOCASE) && c >= 'A' && c <= 'Z' ? c + 32 : c;
    const uint8_t *p = blob + off[u];
    const int32_t *f = pi + off[u];
    uint8_t *rows = dfa + 256ull * off[u];
    int m = (int)(off[u + 1] - off[u]);
    for (int j = 0; j < m; j++) {
        uint8_t entry;
        if (p[j] == fc) entry = (j + 1 == m) ? (uint8_t)(f[m - 1] | 0x80) : (uint8_t)(j + 1);
        else entry = j == 0 ? 0 : rows[256 * f[j - 1] + c]; // mismatch: what the border state does on c
        rows[256 * j + c] = entry;
    }
}

template <typename T>
static int upload(T **dst, const T *src, size_t n, cudaStream_t s)
{
    KMPB_CUDA(cudaMalloc((void **)dst, (n ? n : 1) * sizeof(T)));
    if (n) KMPB_CUDA(cudaMemcpyAsync(*dst, src, n * sizeof(T), cudaMemcpyHostToDevice, s));
    return KMPB_OK;
}

void kmpb_release_tables(kmpb_ctx *ctx)
{
    kmpb_device_tables &d = ctx->dev;
    cudaFree(d.uniq_blob); cudaFree(d.uniq_off); cudaFree(d.uniq_len); cudaFree(d.uniq_flags); cudaFree(d.pat_to_uniq);
    cudaFree(d.pi); cudaFree(d.perpat_dfa); cudaFree(d.filter); cudaFree(d.vtab); cudaFree(d.gate); cudaFree(d.uniq_first);
    cudaFree(d.wvtab); cudaFree(d.uniq_lo); cudaFree(d.uniq_hi);
    d = kmpb_device_tables();
    cudaFree(ctx->d_uniq_counts); ctx->d_uniq_counts = nullptr;
    cudaFree(ctx->d_counts); ctx->d_counts = nullptr;
    if (ctx->have_tables) kmpb_tables_free(&ctx->host);
    ctx->have_tables = false;
}

int kmpb_upload_tables(kmpb_ctx *ctx)
{
    const kmpb_tables &h = ctx->host;
    kmpb_device_tables &d = ctx->dev;
    cudaStream_t s = ctx->stream;
    d.n_pat = h.n_pat; d.n_uniq = h.n_uniq; d.n_class = h.n_class; d.n_state = h.n_state;
    d.max_len = h.max_len; d.min_len = h.min_len;
    size_t blob_len = h.n_uniq ? h.uniq_off[h.n_uniq] : 0;
    int rc;
    if ((rc = upload(&d.uniq_blob, h.uniq_blob, blob_len, s))) return rc;
    if ((rc = upload(&d.uniq_off, h.uniq_off, (size_t)h.n_uniq + 1, s))) return rc;
    if ((rc = upload(&d.uniq_len, h.uniq_len, h.n_uniq, s))) return rc;
    if ((rc = upload(&d.uniq_flags, h.uniq_flags, h.n_uniq, s))) return rc;
    if ((rc = upload(&d.pat_to_uniq, h.pat_to_uniq, h.n_pat, s))) return rc;
    if ((rc = upload(&d.vtab, h.vtab, (size_t)h.vtab_words, s))) return rc;
    if ((rc = upload(&d.filter, h.filter6, 256, s))) return rc;
    if (h.gate_words && (rc = upload(&d.gate, h.gate, h.gate_words, s))) return rc;
    if (h.n_union < h.n_uniq &&
        ((rc = upload(&d.wvtab, h.wvtab, (size_t)h.wvtab_words, s)) || (rc = upload(&d.uniq_lo, h.uniq_lo, h.n_uniq - h.n_union, s)) ||
         (rc = upload(&d.uniq_hi, h.uniq_hi, h.n_uniq - h.n_union, s))))
        return rc;
    {
        uint32_t *first = (uint32_t *)malloc((h.n_uniq ? h.n_uniq : 1) * sizeof(uint32_t));
        if (first == nullptr) return kmpb_fail(KMPB_ENOMEM, "out of memory");
        for (uint32_t i = h.n_pat; i-- > 0;) first[h.pat_to_uniq[i]] = i; // the lowest index is written last
        rc = upload(&d.uniq_first, first, h.n_uniq, s);
        if (rc == KMPB_OK) KMPB_CUDA(cudaStreamSynchronize(s)); // the host table goes away below
        free(first);
        if (rc) return rc;
    }
    KMPB_CUDA(cudaMalloc((void **)&d.pi, (blob_len ? blob_len : 1) * sizeof(int32_t)));
    KMPB_CUDA(cudaMalloc((void **)&d.perpat_dfa, blob_len ? blob_len * 256 : 1));
    // per stream slot: distinct-pattern accumulators
    KMPB_CUDA(cudaMalloc((void **)&ctx->d_uniq_counts, (size_t)KMPB_COPY_STREAMS * (h.n_uniq ? h.n_uniq : 1) * sizeof(uint64_t)));
    KMPB_CUDA(cudaMalloc((void **)&ctx->d_counts, (size_t)(h.n_pat ? h.n_pat : 1) * sizeof(uint64_t)));
    if (h.n_uniq) {
        kmpb_build_prefix_kernel<<<(h.n_uniq + 127) / 128, 128, 0, s>>>(d.uniq_blob, d.uniq_off, h.n_uniq, d.pi);
        kmpb_expand_dfa_kernel<<<h.n_uniq, 256, 0, s>>>(d.uniq_blob, d.uniq_off, d.uniq_flags, d.pi, d.perpat_dfa);
        ctx->launches += 2;
        KMPB_CUDA(cudaGetLastError());
    }
    KMPB_CUDA(cudaStreamSynchronize(s));
    return KMPB_OK;
}
