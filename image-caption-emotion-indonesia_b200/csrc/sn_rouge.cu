// K13: ROUGE-L (DESIGN.md section 4).  Replaces coco-caption's Rouge scorer (pycocoevalcap/rouge/rouge.py,
// Rouge().compute_score): my_lcs and calc_score, on integer token ids.
//
// One warp per image.  The hypothesis (at most SN_BLEU_MAX_LEN tokens) sits in registers: lane l holds position
// 32 w + l in hyp[w].  Each reference is streamed from global memory through the bit-parallel LCS of Crochemore et al.
// (2001) in Hyyro's form, with the hypothesis as the bit side: V starts all ones and, for each reference token y,
//   M = the positions of y in the hypothesis (one __ballot_sync per 32-bit word),  U = V & M,  V = (V + U) | (V - U);
// the LCS length is the number of zero bits of V among the first m (m = hypothesis length).  U is a subset of V, so
// V - U never borrows and only the addition carries from word to word.  Every one of these operations moves information
// from lower bits to higher ones only, so whatever sits at bits >= m (match bits of positions past the hypothesis,
// carries out of bit m - 1) never reaches the first m bits: it is masked off once, when the zeros are counted.
//
// The LCS lengths are exact integers; the score is calc_score's float64 formula, written with __dmul_rn / __dadd_rn /
// __ddiv_rn in its operation order so that nvcc cannot contract any of it into an FMA.  Every operation is then one
// correctly rounded IEEE operation on the same operands as the scorer's, and a score equals the scorer's bit for bit.
// The only reduction is a max; there are no atomics and no float sums.
#include <math.h>

#include "sn_common.cuh"

namespace {

constexpr int kThreads = 128;
constexpr int kWarps = kThreads / 32;
constexpr int kWords = SN_BLEU_MAX_LEN / 32;      // 32-bit words of the bit vector of the longest hypothesis
static_assert(SN_BLEU_MAX_LEN % 32 == 0, "the bit vector is whole 32-bit words");

// bits of word w that stand for hypothesis positions < m
__device__ __forceinline__ uint32_t word_mask(int m, int w) {
  const int k = m - 32 * w;
  return k >= 32 ? ~0u : (k <= 0 ? 0u : (1u << k) - 1u);
}

// LCS length of the hypothesis (m tokens, 1 <= m <= 32 * NW, held as in the file comment) and ref[0 .. n), n >= 1.
// Warp-uniform: every lane returns the same value.
template <int NW>
__device__ __forceinline__ int lcs_bits(const int32_t (&hyp)[kWords], int m, const int32_t* __restrict__ ref, int n,
                                        int lane) {
  uint32_t V[NW];
#pragma unroll
  for (int w = 0; w < NW; ++w) V[w] = ~0u;
  for (int c = 0; c < n; c += 32) {
    const int32_t mine = c + lane < n ? ref[c + lane] : 0;  // 32 reference tokens per coalesced load
    const int k = min(32, n - c);
#pragma unroll 4
    for (int j = 0; j < k; ++j) {
      const int32_t y = __shfl_sync(0xffffffffu, mine, j);
      uint32_t carry = 0;
#pragma unroll
      for (int w = 0; w < NW; ++w) {
        const uint32_t u = V[w] & __ballot_sync(0xffffffffu, hyp[w] == y);
        const uint32_t t = V[w] + u;
        const uint32_t s = t + carry;
        V[w] = s | (V[w] - u);
        carry = (t < u) | (s < t);                            // at most one of the two additions overflows
      }
    }
  }
  int zeros = 0;
#pragma unroll
  for (int w = 0; w < NW; ++w) zeros += __popc(~V[w] & word_mask(m, w));
  return zeros;
}

__device__ __forceinline__ int lcs(const int32_t (&hyp)[kWords], int m, const int32_t* __restrict__ ref, int n,
                                   int lane) {
  switch ((m + 31) >> 5) {                                  // only the words the hypothesis occupies
    case 1: return lcs_bits<1>(hyp, m, ref, n, lane);
    case 2: return lcs_bits<2>(hyp, m, ref, n, lane);
    case 3: return lcs_bits<3>(hyp, m, ref, n, lane);
    case 4: return lcs_bits<4>(hyp, m, ref, n, lane);
    case 5: return lcs_bits<5>(hyp, m, ref, n, lane);
    case 6: return lcs_bits<6>(hyp, m, ref, n, lane);
    case 7: return lcs_bits<7>(hyp, m, ref, n, lane);
    default: return lcs_bits<kWords>(hyp, m, ref, n, lane);
  }
}

// Where hypothesis i comes from.  CSR (kRows = false): hyp_tok[hyp_off[i] .. hyp_off[i + 1]), scored against image i.
// Rows (kRows = true, sampled captions): seqs[i, 1 .. lengths[i]) without a final end_token, scored against image
// img[i] of the corpus (sn_cider.cu's layout).
struct HypRows {
  const int64_t* seqs; int64_t ld; const int64_t* lengths; int32_t end_token; const int64_t* img;
};

// grid (ceil(n_hyp / kWarps)); block kThreads; warp w of CTA b scores hypothesis b * kWarps + w
template <bool kRows>
__global__ void __launch_bounds__(kThreads) rouge_l_kernel(const int32_t* __restrict__ hyp_tok,
                                                           const int64_t* __restrict__ hyp_off, HypRows rows,
                                                           int64_t n_hyp, int64_t n_corpus,
                                                           const int32_t* __restrict__ ref_tok,
                                                           const int64_t* __restrict__ ref_off,
                                                           const int64_t* __restrict__ ref_group, int max_len,
                                                           double beta2, double* __restrict__ scores) {
  const int lane = threadIdx.x & 31;
  const int64_t i = (int64_t)blockIdx.x * kWarps + (threadIdx.x >> 5);
  if (i >= n_hyp) return;                                   // whole warps only
  int64_t h0, L64, gi = i;
  if (kRows) {
    h0 = i * rows.ld + 1;
    L64 = rows.lengths[i] > rows.ld ? -1 : max((int64_t)0, rows.lengths[i] - 1);   // -1: past the row -> NaN below
    if (L64 > 0 && rows.seqs[h0 + L64 - 1] == rows.end_token) --L64;
    gi = rows.img[i];
  } else {
    h0 = hyp_off[i];
    L64 = hyp_off[i + 1] - h0;
  }
  // sizes outside what the caller declared, or an image without references (calc_score asserts len(refs) > 0): NaN
  bool bad = L64 < 0 || L64 > max_len || gi < 0 || gi >= n_corpus;
  const int64_t r0 = bad ? 0 : ref_group[gi], r1 = bad ? 0 : ref_group[gi + 1];
  bad = bad || r1 <= r0;
  for (int64_t r = r0 + lane; r < r1 && !bad; r += 32) bad = ref_off[r + 1] - ref_off[r] > max_len;
  if (__any_sync(0xffffffffu, bad)) {
    if (lane == 0) scores[i] = nan("");
    return;
  }
  const int m = (int)L64;
  int32_t hyp[kWords];
#pragma unroll
  for (int w = 0; w < kWords; ++w) {
    const int p = 32 * w + lane;
    hyp[w] = p < m ? (kRows ? (int32_t)rows.seqs[h0 + p] : hyp_tok[h0 + p]) : 0;
  }
  // "".split(" ") is [""]: an empty sentence is one token, which only another empty sentence has
  int best = 0;                                             // max LCS over the references
  double rec = 0.0;                                         // max over the references of LCS / reference length
  for (int64_t r = r0; r < r1; ++r) {
    const int n = (int)(ref_off[r + 1] - ref_off[r]);
    const int l = (m == 0 || n == 0) ? (m == 0 && n == 0) : lcs(hyp, m, ref_tok + ref_off[r], n, lane);
    best = max(best, l);
    rec = fmax(rec, __ddiv_rn((double)l, (double)max(n, 1)));
  }
  // max over references of LCS / m = (max LCS) / m: correctly rounded division by a positive constant is monotone
  const double prec = __ddiv_rn((double)best, (double)max(m, 1));
  double score = 0.0;
  if (prec != 0.0 && rec != 0.0)                            // ((1 + b2) * p * r) / (r + b2 * p)
    score = __ddiv_rn(__dmul_rn(__dmul_rn(__dadd_rn(1.0, beta2), prec), rec), __dadd_rn(rec, __dmul_rn(beta2, prec)));
  if (lane == 0) scores[i] = score;
}

int32_t check_common(const char* what, int32_t max_sentence_len, double beta2) {
  SN_REQUIRE(max_sentence_len >= 0 && max_sentence_len <= SN_BLEU_MAX_LEN,
             "%s: a sentence has %d tokens; the limit is %d", what, (int)max_sentence_len, SN_BLEU_MAX_LEN);
  SN_REQUIRE(isfinite(beta2) && beta2 >= 0.0, "%s: beta2 = %g must be finite and >= 0", what, beta2);
  return 0;
}

unsigned grid_of(int64_t n) { return (unsigned)((n + kWarps - 1) / kWarps); }

}  // namespace

extern "C" int32_t sn_rouge_l(const int32_t* hyp_tok, const int64_t* hyp_off, int64_t n_img, const int32_t* ref_tok,
                              const int64_t* ref_off, const int64_t* ref_group, int32_t max_sentence_len, double beta2,
                              double* scores, void* stream) {
  SN_REQUIRE(n_img >= 0 && n_img <= 0x7fffffff, "sn_rouge_l: n_img = %lld out of range", (long long)n_img);
  if (int32_t rc = check_common("sn_rouge_l", max_sentence_len, beta2)) return rc;
  if (n_img == 0) return 0;
  SN_REQUIRE(hyp_off && ref_off && ref_group && scores, "sn_rouge_l: null argument");
  rouge_l_kernel<false><<<grid_of(n_img), kThreads, 0, (cudaStream_t)stream>>>(
      hyp_tok, hyp_off, HypRows{}, n_img, n_img, ref_tok, ref_off, ref_group, max_sentence_len, beta2, scores);
  return sn::check_launch("rouge_l_kernel");
}

extern "C" int32_t sn_rouge_l_rows(const int64_t* seqs, int64_t ld, const int64_t* lengths, int64_t R,
                                   int32_t end_token, const int64_t* img, int64_t n_corpus, const int32_t* ref_tok,
                                   const int64_t* ref_off, const int64_t* ref_group, int32_t max_sentence_len,
                                   double beta2, double* scores, void* stream) {
  SN_REQUIRE(R >= 0 && R <= 0x7fffffff, "sn_rouge_l_rows: R = %lld out of range", (long long)R);
  SN_REQUIRE(n_corpus >= 1, "sn_rouge_l_rows: n_corpus = %lld", (long long)n_corpus);
  if (int32_t rc = check_common("sn_rouge_l_rows", max_sentence_len, beta2)) return rc;
  SN_REQUIRE(ld >= 1 && ld - 1 <= max_sentence_len, "sn_rouge_l_rows: ld = %lld does not fit max_sentence_len = %d",
             (long long)ld, (int)max_sentence_len);
  if (R == 0) return 0;
  SN_REQUIRE(seqs && lengths && img && ref_off && ref_group && scores, "sn_rouge_l_rows: null argument");
  rouge_l_kernel<true><<<grid_of(R), kThreads, 0, (cudaStream_t)stream>>>(
      nullptr, nullptr, HypRows{seqs, ld, lengths, end_token, img}, R, n_corpus, ref_tok, ref_off, ref_group,
      max_sentence_len, beta2, scores);
  return sn::check_launch("rouge_l_kernel(rows)");
}
