// Speculative decoding on the paged KV cache: the token history kept next to K / V, n-gram (prompt lookup) drafts from it,
// and the exact acceptance of a verify step's drafts against the tokens the sampler drew for its rows.
//
//   ngram_draft_kernel       one CTA per row: S = the row's history [0, past) read through the block table, then its pending
//                            token.  For n = n_max .. n_min the largest j < |S| - n with S[j, j + n) = the last n tokens of S,
//                            found by a parallel scan and a shared-memory max; the first n that matches proposes S[j + n, ...).
//   speculative_accept_kernel one CTA per row: the leading drafts equal to the sampled token of the row before them are kept,
//                            the kept tokens go to the history pages, and the emitted tokens go to one small output buffer.
// Contract: include/l32_ffn.h (l32_ngram_draft_paged, l32_speculative_accept).
#include "l32_internal.cuh"

namespace l32 {
namespace {

constexpr int kSpecThreads = 256;
constexpr int kPage = L32_KV_PAGE;

// Token i of S: the history up to `past`, then the pending token.
L32_DEVICE int hist_at(const int* __restrict__ pool, const int* __restrict__ table, int past, int pending, int i) {
    return i < past ? __ldg(pool + static_cast<size_t>(__ldg(table + i / kPage)) * kPage + i % kPage) : pending;
}

__global__ void __launch_bounds__(kSpecThreads) ngram_draft_kernel(const int* __restrict__ pool, const int* __restrict__ block_table,
                                                                  const int* __restrict__ past_lens, const long long* __restrict__ pending,
                                                                  long long* __restrict__ ids, int* __restrict__ draft_len, int k,
                                                                  int n_min, int n_max, int max_pages_per_seq) {
    __shared__ int best_j;
    __shared__ int suffix[L32_NGRAM_MAX];
    pdl_wait_prior_grid();
    const int b = blockIdx.x;
    const int past = past_lens[b];
    const int pend = static_cast<int>(pending[b]);
    const int* table = block_table + static_cast<size_t>(b) * max_pages_per_seq;
    const int len = past + 1;                                  // |S|
    int found = -1, n_found = 0;
    for (int n = min(n_max, len - 1); n >= n_min; --n) {
        __syncthreads();                                       // (the previous n's reads of best_j / suffix are done)
        if (threadIdx.x < n) suffix[threadIdx.x] = hist_at(pool, table, past, pend, len - n + threadIdx.x);
        if (threadIdx.x == 0) best_j = -1;
        __syncthreads();
        // candidates j in [0, len - n): the scan runs from the end so that the first match a thread finds is its largest
        for (int j = len - n - 1 - static_cast<int>(threadIdx.x); j >= 0; j -= kSpecThreads) {
            if (j <= *reinterpret_cast<volatile int*>(&best_j)) break;   // (racy: it only skips candidates below a match)
            bool eq = true;
            for (int i = n - 1; i >= 0 && eq; --i) eq = hist_at(pool, table, past, pend, j + i) == suffix[i];
            if (eq) {
                atomicMax(&best_j, j);
                break;
            }
        }
        __syncthreads();
        if (best_j >= 0) {
            found = best_j;
            n_found = n;
            break;
        }
    }
    // ids[b] = pending, then the proposal S[found + n, found + n + k) cut at |S|, padded with its last token (the pending token
    // when there is no proposal)
    long long* row = ids + static_cast<size_t>(b) * (k + 1);
    const int start = found >= 0 ? found + n_found : len;
    const int avail = min(k, len - start);
    for (int i = threadIdx.x; i <= k; i += kSpecThreads) {
        int tok;
        if (i == 0)
            tok = pend;
        else if (i <= avail)
            tok = hist_at(pool, table, past, pend, start + i - 1);
        else
            tok = avail > 0 ? hist_at(pool, table, past, pend, start + avail - 1) : pend;
        row[i] = tok;
    }
    if (threadIdx.x == 0 && draft_len != nullptr) draft_len[b] = avail;
    pdl_launch_dependents();
}

__global__ void __launch_bounds__(kSpecThreads) speculative_accept_kernel(const long long* __restrict__ ids,
                                                                         const long long* __restrict__ sampled, int* __restrict__ pool,
                                                                         const int* __restrict__ block_table,
                                                                         const int* __restrict__ past_lens,
                                                                         const int* __restrict__ new_lens, long long* __restrict__ out,
                                                                         int width, int max_pages_per_seq) {
    __shared__ int acc;
    pdl_wait_prior_grid();
    const int b = blockIdx.x;
    const int n = min(new_lens[b], width);
    if (n <= 0) return;                                        // not in this step: nothing is written
    const long long* row = ids + static_cast<size_t>(b) * width;
    if (threadIdx.x == 0) {
        int a = n;                                             // no sampled tokens: every new token is kept
        if (sampled != nullptr) {
            const long long* s = sampled + static_cast<size_t>(b) * width;
            a = 0;
            while (a < n - 1 && row[a + 1] == s[a]) ++a;
            ++a;                                               // the pending token, then the a - 1 agreeing drafts
        }
        acc = a;
    }
    __syncthreads();
    const int a = acc;
    const int past = past_lens[b];
    const int* table = block_table + static_cast<size_t>(b) * max_pages_per_seq;
    for (int i = threadIdx.x; i < a; i += kSpecThreads) {
        const int pos = past + i;
        pool[static_cast<size_t>(table[pos / kPage]) * kPage + pos % kPage] = static_cast<int>(row[i]);
    }
    if (out != nullptr && sampled != nullptr) {
        long long* o = out + static_cast<size_t>(b) * (width + 1);
        const long long* s = sampled + static_cast<size_t>(b) * width;
        for (int i = threadIdx.x; i <= width; i += kSpecThreads) o[i] = i == 0 ? a : (i <= a ? s[i - 1] : -1ll);
    } else if (out != nullptr && threadIdx.x == 0) {
        out[static_cast<size_t>(b) * (width + 1)] = a;
    }
    pdl_launch_dependents();
}

cudaLaunchConfig_t row_config(int batch, cudaStream_t s, cudaLaunchAttribute* attr) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(static_cast<unsigned>(batch));
    cfg.blockDim = dim3(kSpecThreads);
    cfg.stream = s;
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cfg;
}

}  // namespace

int ngram_draft_paged(const int* token_pool, const int* block_table, const int* past_lens, const long long* pending, long long* ids,
                      int* draft_len, int batch, int k, int n_min, int n_max, int max_pages_per_seq, cudaStream_t s) {
    cudaLaunchAttribute attr[1];
    const cudaLaunchConfig_t cfg = row_config(batch, s, attr);
    const cudaError_t e = cudaLaunchKernelEx(&cfg, ngram_draft_kernel, token_pool, block_table, past_lens, pending, ids, draft_len, k,
                                             n_min, n_max, max_pages_per_seq);
    if (e == cudaSuccess) count_launch();
    return static_cast<int>(e);
}

int speculative_accept(const long long* ids, const long long* sampled, int* token_pool, const int* block_table, const int* past_lens,
                       const int* new_lens, long long* out, int batch, int width, int max_pages_per_seq, cudaStream_t s) {
    cudaLaunchAttribute attr[1];
    const cudaLaunchConfig_t cfg = row_config(batch, s, attr);
    const cudaError_t e = cudaLaunchKernelEx(&cfg, speculative_accept_kernel, ids, sampled, token_pool, block_table, past_lens, new_lens,
                                             out, width, max_pages_per_seq);
    if (e == cudaSuccess) count_launch();
    return static_cast<int>(e);
}

}  // namespace l32
