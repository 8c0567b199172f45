// K12: one step of sampling decode (DESIGN.md section 4) -- the draw of self-critical sequence training.
// One CTA per row makes one pass over the row's logits: the Gumbel-perturbed arg-max (or the plain arg-max) and the
// log-sum-exp of the unscaled logits, then the row's bookkeeping (token, log-probability, length, done flag and the
// count of unfinished rows) -- nothing goes back to the host inside the decode loop.
//
// The noise is a counter-based hash of (seed, step, row, column), restated in numpy by oracle/scst.py: the same seed
// draws the same tokens whatever the launch configuration, and the seed and the step are read from device memory, so
// a step replayed from a CUDA graph draws fresh noise as the step counter moves.
#include <math.h>

#include "sn_common.cuh"

namespace {

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;
constexpr uint64_t kSeedMul = 0x9E3779B97F4A7C15ull;

// the larger of two (score, index) pairs; ties -> the lower index
__device__ __forceinline__ void take_best(double& s, int& i, double os, int oi) {
  if (os > s || (os == s && oi < i)) { s = os; i = oi; }
}

// log-sum-exp accumulator (running max m, sum of exp(x - m))
__device__ __forceinline__ void lse_merge(float& m, float& z, float om, float oz) {
  const float nm = fmaxf(m, om);
  z = (m == -INFINITY ? 0.f : z * expf(m - nm)) + (om == -INFINITY ? 0.f : oz * expf(om - nm));
  m = nm;
}

__global__ void __launch_bounds__(kThreads) sample_step_kernel(
    const float* __restrict__ logits, int64_t ld, int V, int max_len, int end_token, double temperature, int greedy,
    const uint64_t* __restrict__ seed_dev, const int32_t* __restrict__ step_dev, int32_t* __restrict__ prev_word,
    int64_t* __restrict__ seqs, int64_t* __restrict__ lengths, float* __restrict__ logprob, int32_t* __restrict__ done,
    int32_t* __restrict__ n_unfinished) {
  __shared__ double red_s[kWarps];
  __shared__ int red_i[kWarps];
  __shared__ float red_m[kWarps], red_z[kWarps];
  const int r = blockIdx.x;
  if (done[r]) return;                                   // block-uniform
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int step = *step_dev;
  const uint64_t seed_t = *seed_dev * kSeedMul + (uint64_t)step;
  const float* row = logits + (int64_t)r * ld;
  double best = -INFINITY;
  int bi = 0x7fffffff;
  float m = -INFINITY, z = 0.f;
  for (int v = tid; v < V; v += kThreads) {
    const float x = row[v];
    double s = (double)x;
    if (!greedy) {
      const double u = ((double)(sn::hash_u32(seed_t, (uint32_t)r, (uint32_t)v) >> 8) + 0.5) * (1.0 / 16777216.0);
      s = s / temperature - log(-log(u));
    }
    if (s > best) { best = s; bi = v; }                  // strictly greater keeps the lowest index per thread
    if (x > m) { z = (m == -INFINITY ? 0.f : z * expf(m - x)) + 1.f; m = x; }
    else z += expf(x - m);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    take_best(best, bi, __shfl_xor_sync(0xffffffffu, best, o), __shfl_xor_sync(0xffffffffu, bi, o));
    lse_merge(m, z, __shfl_xor_sync(0xffffffffu, m, o), __shfl_xor_sync(0xffffffffu, z, o));
  }
  if (lane == 0) { red_s[warp] = best; red_i[warp] = bi; red_m[warp] = m; red_z[warp] = z; }
  __syncthreads();
  if (tid != 0) return;
  best = red_s[0]; bi = red_i[0]; m = red_m[0]; z = red_z[0];
  for (int w = 1; w < kWarps; ++w) {
    take_best(best, bi, red_s[w], red_i[w]);
    lse_merge(m, z, red_m[w], red_z[w]);
  }
  const int tok = bi;
  const int64_t L = (int64_t)max_len + 2;
  seqs[(int64_t)r * L + step] = tok;
  prev_word[r] = tok;
  logprob[(int64_t)r * (L - 1) + step - 1] = row[tok] - (m + logf(z));
  if (tok == end_token || step == max_len + 1) {
    done[r] = 1;
    lengths[r] = step + 1;
    atomicSub(n_unfinished, 1);
  }
}

}  // namespace

extern "C" int32_t sn_sample_step(const float* logits, int64_t ld, int64_t V, int32_t R, int32_t max_len,
                                  int32_t end_token, double temperature, int32_t greedy, const uint64_t* seed_dev,
                                  const int32_t* step_dev, int32_t* prev_word, int64_t* seqs, int64_t* lengths,
                                  float* logprob, int32_t* done, int32_t* n_unfinished, void* stream) {
  SN_REQUIRE(R >= 0 && V > 0 && V <= 0x7fffffff && ld >= V && max_len >= 0, "sn_sample_step: bad dims");
  SN_REQUIRE(greedy || (isfinite(temperature) && temperature > 0.0),
             "sn_sample_step: temperature = %g must be finite and > 0", temperature);
  if (R == 0) return 0;
  SN_REQUIRE(logits && seed_dev && step_dev && prev_word && seqs && lengths && logprob && done && n_unfinished,
             "sn_sample_step: null argument");
  sample_step_kernel<<<(unsigned)R, kThreads, 0, (cudaStream_t)stream>>>(logits, ld, (int)V, max_len, end_token,
                                                                         temperature, greedy, seed_dev, step_dev,
                                                                         prev_word, seqs, lengths, logprob, done,
                                                                         n_unfinished);
  return sn::check_launch("sample_step_kernel");
}
