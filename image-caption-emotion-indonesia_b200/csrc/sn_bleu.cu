// K10: corpus-BLEU n-gram statistics (DESIGN.md section 4).  Replaces the per-hypothesis loop of nltk's corpus_bleu --
// modified_precision and closest_ref_length (nltk/translate/bleu_score.py) -- that the reference runs at the end of
// every validation epoch (stylenet/train_multitask.py:341, evaluator.py:103).
//
// One CTA per hypothesis.  The hypothesis and its references are staged in shared memory; a thread owns (order n,
// position p) pairs.  The n-gram g starting at p is counted only where it occurs first in the hypothesis, so every
// distinct n-gram contributes once: min(count_hyp(g), max over refs of count_ref(g)).  Tokens are compared directly,
// nothing is hashed.  Integer arithmetic only, no atomics: the statistics are exact and identical on every run.
#include "sn_common.cuh"

namespace {

constexpr int kThreads = 128;
constexpr int kMaxOrder = 4;

// occurrences of the n-gram g[0..n) in s[0..m)
__device__ __forceinline__ int count_ngram(const int32_t* s, int m, const int32_t (&g)[kMaxOrder], int n) {
  int c = 0;
  for (int q = 0; q + n <= m; ++q) {
    bool eq = s[q] == g[0];
    for (int k = 1; k < n && eq; ++k) eq = s[q + k] == g[k];
    c += eq;
  }
  return c;
}

// grid (n_hyp); block kThreads; dynamic shared memory: cap_tokens int32
__global__ void __launch_bounds__(kThreads) bleu_counts_kernel(const int32_t* __restrict__ hyp_tok,
                                                               const int64_t* __restrict__ hyp_off,
                                                               const int32_t* __restrict__ ref_tok,
                                                               const int64_t* __restrict__ ref_off,
                                                               const int64_t* __restrict__ ref_group, int max_len,
                                                               int64_t cap_tokens, int32_t* __restrict__ stats) {
  extern __shared__ int32_t tok[];              // [hypothesis | reference 0 | reference 1 | ...]
  __shared__ int32_t part[kThreads / 32][kMaxOrder];
  const int i = blockIdx.x;
  const int64_t h0 = hyp_off[i], r0 = ref_group[i], r1 = ref_group[i + 1];
  const int64_t L64 = hyp_off[i + 1] - h0;
  const int64_t base = ref_off[r0], nref_tok = ref_off[r1] - base;
  int32_t* out = stats + (int64_t)i * 10;
  // sizes larger than the caller declared: every column -1, nothing read past the staging buffer
  bool bad = L64 < 0 || L64 > max_len || nref_tok < 0 || L64 + nref_tok > cap_tokens;
  for (int64_t r = r0; r < r1 && !bad; ++r) bad = ref_off[r + 1] - ref_off[r] > max_len;
  if (bad) {
    if (threadIdx.x < 10) out[threadIdx.x] = -1;
    return;
  }
  const int L = (int)L64;
  const int nr = (int)nref_tok;
  for (int t = threadIdx.x; t < L; t += kThreads) tok[t] = hyp_tok[h0 + t];
  for (int t = threadIdx.x; t < nr; t += kThreads) tok[L + t] = ref_tok[base + t];
  __syncthreads();
  const int32_t* hyp = tok;
  const int32_t* refs = tok + L;

  int acc[kMaxOrder] = {0, 0, 0, 0};
  for (int j = threadIdx.x; j < kMaxOrder * L; j += kThreads) {
    const int n = j / L + 1, p = j - (n - 1) * L;
    if (p + n > L) continue;
    int32_t g[kMaxOrder];
#pragma unroll
    for (int k = 0; k < kMaxOrder; ++k) g[k] = k < n ? hyp[p + k] : 0;
    if (count_ngram(hyp, p + n - 1, g, n) > 0) continue;   // not the first occurrence
    const int ch = count_ngram(hyp + p, L - p, g, n);      // first occurrence: later ones are all after p
    int mx = 0;
    for (int64_t r = r0; r < r1 && mx < ch; ++r) {
      const int s = (int)(ref_off[r] - base), m = (int)(ref_off[r + 1] - ref_off[r]);
      mx = max(mx, count_ngram(refs + s, m, g, n));
    }
    const int clipped = min(ch, mx);
#pragma unroll
    for (int k = 0; k < kMaxOrder; ++k) acc[k] += (k == n - 1) ? clipped : 0;
  }
  // block reduction in a fixed order: warp shuffles, then warp 0 over the per-warp partials
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < kMaxOrder; ++k) {
    int v = acc[k];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (lane == 0) part[warp][k] = v;
  }
  __syncthreads();
  if (threadIdx.x < kMaxOrder) {
    int v = 0;
    for (int w = 0; w < kThreads / 32; ++w) v += part[w][threadIdx.x];
    out[threadIdx.x] = v;                                  // clipped matches, order threadIdx.x + 1
    out[kMaxOrder + threadIdx.x] = max(1, L - (int)threadIdx.x);   // max(1, L - n + 1)
  } else if (threadIdx.x == kMaxOrder) {
    out[8] = L;
  } else if (threadIdx.x == kMaxOrder + 1) {
    // closest reference length: minimise (|len_ref - L|, len_ref); 0 when there is no reference
    int best = 0, best_d = -1;
    for (int64_t r = r0; r < r1; ++r) {
      const int m = (int)(ref_off[r + 1] - ref_off[r]), d = abs(m - L);
      if (best_d < 0 || d < best_d || (d == best_d && m < best)) best = m, best_d = d;
    }
    out[9] = best;
  }
}

}  // namespace

extern "C" int32_t sn_bleu_counts(const int32_t* hyp_tok, const int64_t* hyp_off, int64_t n_hyp,
                                  const int32_t* ref_tok, const int64_t* ref_off, const int64_t* ref_group,
                                  int32_t max_sentence_len, int64_t max_group_tokens, int32_t* stats, void* stream) {
  SN_REQUIRE(n_hyp >= 0 && n_hyp <= 0x7fffffff, "sn_bleu_counts: n_hyp = %lld out of range", (long long)n_hyp);
  SN_REQUIRE(max_sentence_len >= 0 && max_sentence_len <= SN_BLEU_MAX_LEN,
             "sn_bleu_counts: a sentence has %d tokens; the limit is %d", (int)max_sentence_len, SN_BLEU_MAX_LEN);
  SN_REQUIRE(max_group_tokens >= 0, "sn_bleu_counts: max_group_tokens = %lld", (long long)max_group_tokens);
  if (n_hyp == 0) return 0;
  SN_REQUIRE(hyp_off && ref_off && ref_group && stats, "sn_bleu_counts: null argument");
  const int64_t smem = max_group_tokens * (int64_t)sizeof(int32_t);
  const int optin = sn::dev_info().smem_optin;
  SN_REQUIRE(smem + (int64_t)sizeof(int32_t) * (kThreads / 32) * kMaxOrder <= optin,
             "sn_bleu_counts: a hypothesis and its references hold %lld tokens; at most %lld fit in shared memory",
             (long long)max_group_tokens, (long long)(optin / (int64_t)sizeof(int32_t) - (kThreads / 32) * kMaxOrder));
  if (smem > 48 * 1024)
    SN_CUDA(cudaFuncSetAttribute(bleu_counts_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  bleu_counts_kernel<<<(unsigned)n_hyp, kThreads, (size_t)smem, (cudaStream_t)stream>>>(
      hyp_tok, hyp_off, ref_tok, ref_off, ref_group, max_sentence_len, max_group_tokens, stats);
  return sn::check_launch("bleu_counts_kernel");
}
