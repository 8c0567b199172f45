// K11: CIDEr-D (DESIGN.md section 4).  Replaces coco-caption's CiderScorer (pycocoevalcap/cider/cider_scorer.py):
// compute_doc_freq is sn_cider_df, counts2vec + sim + the per-image mean of compute_cider are sn_cider_scores.
//
// Unlike BLEU (K10), CIDEr-D weights every n-gram by its document frequency over the references of the whole corpus,
// so the first kernel fills a corpus-wide table on the device and the second reads it.  The table is open addressing
// with linear probing on the full key (order + up to 4 ids, one 16-byte slot): a 128-bit compare-and-swap claims an
// empty slot or returns the key already there, so two n-grams can never share a slot whatever their hash, and counts
// are int32 atomic adds (exact, independent of launch order).
//
// Both kernels use one CTA per image with its sentences staged in shared memory, as K10 does, and count an n-gram at
// its first occurrence only.  The scores are float64 throughout; every sum runs in an order fixed by the launch
// configuration (per-thread partials, warp butterflies, warps in index order), with no float atomics.
#include <math.h>

#include "sn_common.cuh"

namespace {

constexpr int kMaxOrder = 4;
constexpr int kDfThreads = 128;
constexpr int kScoreThreads = 256;
constexpr int kScoreWarps = kScoreThreads / 32;
constexpr uint64_t kEmpty = ~0ull;          // an empty slot: four -1 ids (a key's first id is >= 0)

constexpr int32_t kErrFull = 1, kErrNegativeId = 2, kErrSizes = 4;

// the n-gram of order n at s[0..n): ids in the low words first, -1 past the order (little-endian int32 [4] in memory)
__device__ __forceinline__ void make_key(const int32_t* s, int n, uint64_t& lo, uint64_t& hi) {
  uint32_t w[kMaxOrder];
#pragma unroll
  for (int k = 0; k < kMaxOrder; ++k) w[k] = k < n ? (uint32_t)s[k] : 0xffffffffu;
  lo = (uint64_t)w[0] | (uint64_t)w[1] << 32;
  hi = (uint64_t)w[2] | (uint64_t)w[3] << 32;
}

__device__ __forceinline__ uint64_t first_slot(uint64_t lo, uint64_t hi, uint64_t mask) {
  uint64_t x = lo * 0x9e3779b97f4a7c15ull ^ (hi + 0x632be59bd9b4e019ull);
  x ^= x >> 31; x *= 0xbf58476d1ce4e5b9ull;
  x ^= x >> 29; x *= 0x94d049bb133111ebull;
  x ^= x >> 32;
  return x & mask;
}

// 128-bit compare-and-swap (sm_90+): returns the slot's previous contents
__device__ __forceinline__ void cas128(uint64_t* slot, uint64_t cmp_lo, uint64_t cmp_hi, uint64_t lo, uint64_t hi,
                                       uint64_t& old_lo, uint64_t& old_hi) {
  asm volatile(
      "{\n\t.reg .b128 c, v, o;\n\t"
      "mov.b128 c, {%2, %3};\n\t"
      "mov.b128 v, {%4, %5};\n\t"
      "atom.relaxed.gpu.global.cas.b128 o, [%6], c, v;\n\t"
      "mov.b128 {%0, %1}, o;\n\t}"
      : "=l"(old_lo), "=l"(old_hi)
      : "l"(cmp_lo), "l"(cmp_hi), "l"(lo), "l"(hi), "l"(slot)
      : "memory");
}

// ids equal over n positions
__device__ __forceinline__ bool same(const int32_t* a, const int32_t* b, int n) {
  bool eq = true;
  for (int k = 0; k < n && eq; ++k) eq = a[k] == b[k];
  return eq;
}

// occurrences of the n-gram g[0..n) in s[0..m)
__device__ __forceinline__ int count_ngram(const int32_t* s, int m, const int32_t* g, int n) {
  int c = 0;
  for (int q = 0; q + n <= m; ++q) c += same(s + q, g, n);
  return c;
}

// document frequency of a key: its count, 0 when an empty slot (or a whole table without it) ends the probe chain
__device__ __forceinline__ int df_lookup(const ulonglong2* __restrict__ keys, const int32_t* __restrict__ counts,
                                         uint64_t mask, uint64_t lo, uint64_t hi) {
  uint64_t s = first_slot(lo, hi, mask);
  for (uint64_t probe = 0; probe <= mask; ++probe, s = (s + 1) & mask) {
    const ulonglong2 k = keys[s];
    if (k.x == lo && k.y == hi) return counts[s];
    if (k.x == kEmpty && k.y == kEmpty) return 0;
  }
  return 0;
}

__device__ __forceinline__ double idf_of(double ref_len, int df) { return ref_len - log(fmax(1.0, (double)df)); }

// grid (n_img); block kDfThreads; dynamic shared memory: cap_tokens int32 ids, then cap_tokens uint16
__global__ void __launch_bounds__(kDfThreads) cider_df_kernel(const int32_t* __restrict__ ref_tok,
                                                              const int64_t* __restrict__ ref_off,
                                                              const int64_t* __restrict__ ref_group, int n,
                                                              int max_len, int64_t cap_tokens, uint64_t* keys,
                                                              int32_t* counts, uint64_t mask, int32_t* err) {
  extern __shared__ int32_t tok[];                         // [reference 0 | reference 1 | ...]
  uint16_t* rem = reinterpret_cast<uint16_t*>(tok + cap_tokens);   // ids left in its reference from this one on
  const int i = blockIdx.x;
  const int64_t r0 = ref_group[i], r1 = ref_group[i + 1];
  const int64_t base = ref_off[r0], total = ref_off[r1] - base;
  bool bad = total < 0 || total > cap_tokens;
  for (int64_t r = r0; r < r1 && !bad; ++r) bad = ref_off[r + 1] - ref_off[r] > max_len;
  if (bad) {
    if (threadIdx.x == 0) atomicOr(err, kErrSizes);
    return;
  }
  const int T = (int)total;
  for (int t = threadIdx.x; t < T; t += kDfThreads) tok[t] = ref_tok[base + t];
  for (int64_t r = r0; r < r1; ++r) {
    const int s = (int)(ref_off[r] - base), m = (int)(ref_off[r + 1] - ref_off[r]);
    for (int p = threadIdx.x; p < m; p += kDfThreads) rem[s + p] = (uint16_t)(m - p);
  }
  __syncthreads();
  // item j = (order k + 1, start t in the concatenated references); an n-gram may not run past its reference's end
  for (int j = threadIdx.x; j < n * T; j += kDfThreads) {
    const int k = j / T, t = j - k * T, len = k + 1;
    if (rem[t] < len) continue;
    bool seen = false;                                     // an earlier occurrence in this image's references
    for (int q = 0; q < t && !seen; ++q) seen = rem[q] >= len && same(tok + q, tok + t, len);
    if (seen) continue;
    bool negative = false;
    for (int w = 0; w < len; ++w) negative |= tok[t + w] < 0;
    if (negative) {
      atomicOr(err, kErrNegativeId);
      continue;
    }
    uint64_t lo, hi;
    make_key(tok + t, len, lo, hi);
    uint64_t s = first_slot(lo, hi, mask);
    bool placed = false;
    for (uint64_t probe = 0; probe <= mask; ++probe, s = (s + 1) & mask) {
      uint64_t olo, ohi;
      cas128(keys + 2 * s, kEmpty, kEmpty, lo, hi, olo, ohi);
      if ((olo == kEmpty && ohi == kEmpty) || (olo == lo && ohi == hi)) {
        atomicAdd(counts + s, 1);
        placed = true;
        break;
      }
    }
    if (!placed) atomicOr(err, kErrFull);
  }
}

// v[k] += x for a 4-vector held in registers (k is not a compile-time constant).  The products and sums of the scores
// use __dmul_rn / __dadd_rn so that nvcc does not contract them into FMAs: each rounds once, as in the scorer.
__device__ __forceinline__ void add_at(double (&v)[kMaxOrder], int k, double x) {
#pragma unroll
  for (int q = 0; q < kMaxOrder; ++q)
    if (q == k) v[q] = __dadd_rn(v[q], x);
}

__device__ __forceinline__ double warp_sum_f64(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Where hypothesis i comes from.  CSR (kRows = false): hyp_tok[hyp_off[i] .. hyp_off[i + 1]), scored against image i.
// Rows (kRows = true, sampled captions): seqs[i, 1 .. lengths[i]) without a final end_token, scored against image
// img[i] of the corpus.
struct HypRows {
  const int64_t* seqs; int64_t ld; const int64_t* lengths; int32_t end_token; const int64_t* img;
};

// grid (number of hypotheses); block kScoreThreads; dynamic shared memory: kMaxOrder * max_len doubles (idf of the
// hypothesis n-grams), kMaxOrder * max_len int32 (their tf, 0 where the n-gram is not a first occurrence), cap_tokens
// int32 ids.  ref_len = log(n_corpus).
template <bool kRows>
__global__ void __launch_bounds__(kScoreThreads, kRows ? 1 : 0) cider_scores_kernel(
    const int32_t* __restrict__ hyp_tok, const int64_t* __restrict__ hyp_off, HypRows rows, int64_t n_corpus,
    const int32_t* __restrict__ ref_tok,
    const int64_t* __restrict__ ref_off, const int64_t* __restrict__ ref_group, int n, double sigma, int max_len,
    int64_t cap_tokens, const ulonglong2* __restrict__ keys, const int32_t* __restrict__ counts, uint64_t mask,
    double* __restrict__ scores, double* __restrict__ per_order) {
  extern __shared__ double hidf[];                         // [kMaxOrder * max_len]
  int32_t* htf = reinterpret_cast<int32_t*>(hidf + kMaxOrder * max_len);
  int32_t* tok = htf + kMaxOrder * max_len;                // [hypothesis | reference 0 | reference 1 | ...]
  __shared__ double part_h[kScoreWarps][kMaxOrder];
  __shared__ double part_s[kScoreWarps][kMaxOrder];
  const int i = blockIdx.x;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int64_t h0, L64, gi = i;
  if (kRows) {
    h0 = (int64_t)i * rows.ld + 1;
    L64 = rows.lengths[i] > rows.ld ? -1 : max((int64_t)0, rows.lengths[i] - 1);   // -1: past the row -> NaN below
    if (L64 > 0 && rows.seqs[h0 + L64 - 1] == rows.end_token) --L64;
    gi = rows.img[i];
  } else {
    h0 = hyp_off[i];
    L64 = hyp_off[i + 1] - h0;
  }
  const int64_t r0 = ref_group[gi], r1 = ref_group[gi + 1];
  const int64_t base = ref_off[r0], nref_tok = ref_off[r1] - base;
  bool bad = L64 < 0 || L64 > max_len || nref_tok < 0 || L64 + nref_tok > cap_tokens;
  for (int64_t r = r0; r < r1 && !bad; ++r) bad = ref_off[r + 1] - ref_off[r] > max_len;
  if (bad) {
    if (threadIdx.x == 0) scores[i] = nan("");
    if (per_order && threadIdx.x < kMaxOrder) per_order[(int64_t)i * kMaxOrder + threadIdx.x] = nan("");
    return;
  }
  const int L = (int)L64;
  const int nr = (int)nref_tok;
  for (int t = threadIdx.x; t < L; t += kScoreThreads) tok[t] = kRows ? (int32_t)rows.seqs[h0 + t] : hyp_tok[h0 + t];
  for (int t = threadIdx.x; t < nr; t += kScoreThreads) tok[L + t] = ref_tok[base + t];
  __syncthreads();
  const int32_t* hyp = tok;
  const int32_t* refs = tok + L;
  const double ref_len = log((double)n_corpus);

  // counts2vec of the hypothesis: tf and idf at the first occurrence of each n-gram, the squared norm per order
  double nh[kMaxOrder] = {0.0, 0.0, 0.0, 0.0};
  for (int j = threadIdx.x; j < n * L; j += kScoreThreads) {
    const int k = j / L, p = j - k * L, len = k + 1;
    int tf = 0;
    if (p + len <= L && count_ngram(hyp, p + len - 1, hyp + p, len) == 0) {
      tf = count_ngram(hyp + p, L - p, hyp + p, len);
      uint64_t lo, hi;
      make_key(hyp + p, len, lo, hi);
      const double idf = idf_of(ref_len, df_lookup(keys, counts, mask, lo, hi));
      const double v = (double)tf * idf;
      add_at(nh, k, __dmul_rn(v, v));
      hidf[j] = idf;
    }
    htf[j] = tf;
  }
#pragma unroll
  for (int k = 0; k < kMaxOrder; ++k) {
    const double v = warp_sum_f64(nh[k]);
    if (lane == 0) part_h[warp][k] = v;
  }
  __syncthreads();
  double norm_h[kMaxOrder];
#pragma unroll
  for (int k = 0; k < kMaxOrder; ++k) {
    double v = 0.0;
    for (int w = 0; w < kScoreWarps; ++w) v += part_h[w][k];
    norm_h[k] = sqrt(v);
  }
  const int length_h = n >= 2 ? max(0, L - 1) : 0;

  // sim against each reference: warp w takes references w, w + kScoreWarps, ... and keeps their sum per order
  double acc[kMaxOrder] = {0.0, 0.0, 0.0, 0.0};
  for (int64_t r = r0 + warp; r < r1; r += kScoreWarps) {
    const int32_t* ref = refs + (ref_off[r] - base);
    const int m = (int)(ref_off[r + 1] - ref_off[r]);
    const int length_r = n >= 2 ? max(0, m - 1) : 0;
    const double delta = (double)(length_h - length_r);
    const double penalty = pow(2.718281828459045, -(delta * delta) / (2.0 * (sigma * sigma)));   // np.e ** x
    double nr2[kMaxOrder] = {0.0, 0.0, 0.0, 0.0};
    double val[kMaxOrder] = {0.0, 0.0, 0.0, 0.0};
    for (int j = lane; j < n * m; j += 32) {             // counts2vec of the reference: its squared norm per order
      const int k = j / m, p = j - k * m, len = k + 1;
      if (p + len > m || count_ngram(ref, p + len - 1, ref + p, len) != 0) continue;
      const int tf = count_ngram(ref + p, m - p, ref + p, len);
      uint64_t lo, hi;
      make_key(ref + p, len, lo, hi);
      const double v = (double)tf * idf_of(ref_len, df_lookup(keys, counts, mask, lo, hi));
      add_at(nr2, k, __dmul_rn(v, v));
    }
    for (int j = lane; j < n * L; j += 32) {             // clipped products over the hypothesis n-grams
      const int tf = htf[j];
      if (tf == 0) continue;
      const int k = j / L, p = j - k * L;
      const int tfr = count_ngram(ref, m, hyp + p, k + 1);
      if (tfr == 0) continue;
      const double vh = (double)tf * hidf[j], vr = (double)tfr * hidf[j];
      add_at(val, k, __dmul_rn(fmin(vh, vr), vr));
    }
#pragma unroll
    for (int k = 0; k < kMaxOrder; ++k) {
      const double norm_r = sqrt(warp_sum_f64(nr2[k]));
      double v = warp_sum_f64(val[k]);
      if (norm_h[k] != 0.0 && norm_r != 0.0) v /= norm_h[k] * norm_r;
      acc[k] = __dadd_rn(acc[k], __dmul_rn(v, penalty));
    }
  }
  if (lane == 0) {
#pragma unroll
    for (int k = 0; k < kMaxOrder; ++k) part_s[warp][k] = acc[k];
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    double mean = 0.0;
    for (int k = 0; k < kMaxOrder; ++k) {
      double v = 0.0;
      for (int w = 0; w < kScoreWarps; ++w) v += part_s[w][k];
      if (per_order) per_order[(int64_t)i * kMaxOrder + k] = k < n ? v : 0.0;
      if (k < n) mean += v;
    }
    scores[i] = mean / n / (double)(r1 - r0) * 10.0;
  }
}

}  // namespace

extern "C" int32_t sn_cider_df(const int32_t* ref_tok, const int64_t* ref_off, const int64_t* ref_group,
                               int64_t n_img, int32_t n, int32_t max_sentence_len, int64_t max_group_tokens,
                               int32_t* keys, int32_t* counts, int64_t capacity, int32_t* err, void* stream) {
  SN_REQUIRE(n_img >= 0 && n_img <= 0x7fffffff, "sn_cider_df: n_img = %lld out of range", (long long)n_img);
  SN_REQUIRE(n >= 1 && n <= kMaxOrder, "sn_cider_df: n = %d; orders 1..%d are supported", (int)n, kMaxOrder);
  SN_REQUIRE(max_sentence_len >= 0 && max_sentence_len <= SN_BLEU_MAX_LEN,
             "sn_cider_df: a sentence has %d tokens; the limit is %d", (int)max_sentence_len, SN_BLEU_MAX_LEN);
  SN_REQUIRE(max_group_tokens >= 0, "sn_cider_df: max_group_tokens = %lld", (long long)max_group_tokens);
  SN_REQUIRE(capacity > 0 && (capacity & (capacity - 1)) == 0,
             "sn_cider_df: capacity = %lld is not a power of two", (long long)capacity);
  SN_REQUIRE(keys && counts && err, "sn_cider_df: null table argument");
  SN_REQUIRE(((uintptr_t)keys & 15) == 0, "sn_cider_df: keys must be 16-byte aligned");
  const int64_t smem = max_group_tokens * (int64_t)(sizeof(int32_t) + sizeof(uint16_t));
  const int optin = sn::dev_info().smem_optin;
  SN_REQUIRE(smem <= optin,
             "sn_cider_df: the references of an image hold %lld tokens; at most %lld fit in shared memory",
             (long long)max_group_tokens, (long long)(optin / (int64_t)(sizeof(int32_t) + sizeof(uint16_t))));
  cudaStream_t s = (cudaStream_t)stream;
  SN_CUDA(cudaMemsetAsync(keys, 0xff, (size_t)capacity * 4 * sizeof(int32_t), s));
  SN_CUDA(cudaMemsetAsync(counts, 0, (size_t)capacity * sizeof(int32_t), s));
  SN_CUDA(cudaMemsetAsync(err, 0, sizeof(int32_t), s));
  if (n_img == 0) return 0;
  SN_REQUIRE(ref_off && ref_group, "sn_cider_df: null argument");
  if (smem > 48 * 1024)
    SN_CUDA(cudaFuncSetAttribute(cider_df_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  cider_df_kernel<<<(unsigned)n_img, kDfThreads, (size_t)smem, s>>>(ref_tok, ref_off, ref_group, n, max_sentence_len,
                                                                    max_group_tokens, (uint64_t*)keys, counts,
                                                                    (uint64_t)capacity - 1, err);
  return sn::check_launch("cider_df_kernel");
}

extern "C" int32_t sn_cider_scores(const int32_t* hyp_tok, const int64_t* hyp_off, int64_t n_img,
                                   const int32_t* ref_tok, const int64_t* ref_off, const int64_t* ref_group,
                                   int32_t n, double sigma, int32_t max_sentence_len, int64_t max_group_tokens,
                                   const int32_t* keys, const int32_t* counts, int64_t capacity, double* scores,
                                   double* per_order, void* stream) {
  SN_REQUIRE(n_img >= 0 && n_img <= 0x7fffffff, "sn_cider_scores: n_img = %lld out of range", (long long)n_img);
  SN_REQUIRE(n >= 1 && n <= kMaxOrder, "sn_cider_scores: n = %d; orders 1..%d are supported", (int)n, kMaxOrder);
  SN_REQUIRE(isfinite(sigma) && sigma > 0.0, "sn_cider_scores: sigma = %g must be finite and > 0", sigma);
  SN_REQUIRE(max_sentence_len >= 0 && max_sentence_len <= SN_BLEU_MAX_LEN,
             "sn_cider_scores: a sentence has %d tokens; the limit is %d", (int)max_sentence_len, SN_BLEU_MAX_LEN);
  SN_REQUIRE(max_group_tokens >= 0, "sn_cider_scores: max_group_tokens = %lld", (long long)max_group_tokens);
  SN_REQUIRE(capacity > 0 && (capacity & (capacity - 1)) == 0,
             "sn_cider_scores: capacity = %lld is not a power of two", (long long)capacity);
  if (n_img == 0) return 0;
  SN_REQUIRE(hyp_off && ref_off && ref_group && keys && counts && scores, "sn_cider_scores: null argument");
  SN_REQUIRE(((uintptr_t)keys & 15) == 0, "sn_cider_scores: keys must be 16-byte aligned");
  const int64_t hyp_bytes = (int64_t)kMaxOrder * max_sentence_len * (int64_t)(sizeof(double) + sizeof(int32_t));
  const int64_t smem = hyp_bytes + max_group_tokens * (int64_t)sizeof(int32_t);
  const int64_t static_smem = 2 * kScoreWarps * kMaxOrder * (int64_t)sizeof(double);
  const int optin = sn::dev_info().smem_optin;
  SN_REQUIRE(smem + static_smem <= optin,
             "sn_cider_scores: a hypothesis and its references hold %lld tokens; at most %lld fit in shared memory",
             (long long)max_group_tokens, (long long)((optin - static_smem - hyp_bytes) / (int64_t)sizeof(int32_t)));
  if (smem > 48 * 1024)
    SN_CUDA(cudaFuncSetAttribute(cider_scores_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  cider_scores_kernel<false><<<(unsigned)n_img, kScoreThreads, (size_t)smem, (cudaStream_t)stream>>>(
      hyp_tok, hyp_off, HypRows{}, n_img, ref_tok, ref_off, ref_group, n, sigma, max_sentence_len, max_group_tokens,
      reinterpret_cast<const ulonglong2*>(keys), counts, (uint64_t)capacity - 1, scores, per_order);
  return sn::check_launch("cider_scores_kernel");
}

extern "C" int32_t sn_cider_scores_rows(const int64_t* seqs, int64_t ld, const int64_t* lengths, int64_t R,
                                        int32_t end_token, const int64_t* img, int64_t n_corpus, const int32_t* ref_tok,
                                        const int64_t* ref_off, const int64_t* ref_group, int32_t n, double sigma,
                                        int32_t max_sentence_len, int64_t max_group_tokens, const int32_t* keys,
                                        const int32_t* counts, int64_t capacity, double* scores, void* stream) {
  SN_REQUIRE(R >= 0 && R <= 0x7fffffff, "sn_cider_scores_rows: R = %lld out of range", (long long)R);
  SN_REQUIRE(n_corpus >= 1, "sn_cider_scores_rows: n_corpus = %lld", (long long)n_corpus);
  SN_REQUIRE(ld >= 1 && ld - 1 <= max_sentence_len, "sn_cider_scores_rows: ld = %lld does not fit max_sentence_len = %d",
             (long long)ld, (int)max_sentence_len);
  SN_REQUIRE(max_group_tokens >= ld - 1, "sn_cider_scores_rows: max_group_tokens = %lld < ld - 1",
             (long long)max_group_tokens);
  SN_REQUIRE(n >= 1 && n <= kMaxOrder, "sn_cider_scores_rows: n = %d; orders 1..%d are supported", (int)n, kMaxOrder);
  SN_REQUIRE(isfinite(sigma) && sigma > 0.0, "sn_cider_scores_rows: sigma = %g must be finite and > 0", sigma);
  SN_REQUIRE(max_sentence_len >= 0 && max_sentence_len <= SN_BLEU_MAX_LEN,
             "sn_cider_scores_rows: a sentence has %d tokens; the limit is %d", (int)max_sentence_len, SN_BLEU_MAX_LEN);
  SN_REQUIRE(capacity > 0 && (capacity & (capacity - 1)) == 0,
             "sn_cider_scores_rows: capacity = %lld is not a power of two", (long long)capacity);
  if (R == 0) return 0;
  SN_REQUIRE(seqs && lengths && img && ref_off && ref_group && keys && counts && scores,
             "sn_cider_scores_rows: null argument");
  SN_REQUIRE(((uintptr_t)keys & 15) == 0, "sn_cider_scores_rows: keys must be 16-byte aligned");
  const int64_t hyp_bytes = (int64_t)kMaxOrder * max_sentence_len * (int64_t)(sizeof(double) + sizeof(int32_t));
  const int64_t smem = hyp_bytes + max_group_tokens * (int64_t)sizeof(int32_t);
  const int64_t static_smem = 2 * kScoreWarps * kMaxOrder * (int64_t)sizeof(double);
  const int optin = sn::dev_info().smem_optin;
  SN_REQUIRE(smem + static_smem <= optin,
             "sn_cider_scores_rows: a hypothesis and its references hold %lld tokens; at most %lld fit in shared memory",
             (long long)max_group_tokens, (long long)((optin - static_smem - hyp_bytes) / (int64_t)sizeof(int32_t)));
  if (smem > 48 * 1024)
    SN_CUDA(cudaFuncSetAttribute(cider_scores_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  cider_scores_kernel<true><<<(unsigned)R, kScoreThreads, (size_t)smem, (cudaStream_t)stream>>>(
      nullptr, nullptr, HypRows{seqs, ld, lengths, end_token, img}, n_corpus, ref_tok, ref_off, ref_group, n, sigma,
      max_sentence_len, max_group_tokens, reinterpret_cast<const ulonglong2*>(keys), counts, (uint64_t)capacity - 1,
      scores, nullptr);
  return sn::check_launch("cider_scores_kernel(rows)");
}
