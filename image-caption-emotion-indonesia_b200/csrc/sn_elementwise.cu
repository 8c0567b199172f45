#include <stdlib.h>
#include <string.h>
// Memory-bound kernels of the hot path: K1 gather/dropout/pack, K5 log-softmax+NLL(+grad, argmax,
// top-5), deterministic loss reduction, K7 fused clamp+Adam.  All HBM-bound: coalesced, 16-byte
// vectorised where the layout allows, grids sized from the SM count.
#include <cuda_bf16.h>

#include "sn_common.cuh"

namespace {

// ------------------------------------------------------------------------------------------
// K1
// ------------------------------------------------------------------------------------------
__global__ void gather_pack_fwd_kernel(const int64_t* __restrict__ captions, int64_t cap_ld,
                                       const float* __restrict__ table, int E,
                                       const float* __restrict__ features, int64_t feat_ld, int has_feat,
                                       const int32_t* __restrict__ row_b, const int32_t* __restrict__ row_t,
                                       const int32_t* __restrict__ tok_override, int64_t N,
                                       float* __restrict__ X, int64_t ldx, float p, float inv_keep,
                                       uint64_t seed, const uint64_t* __restrict__ seed_dev,
                                       __nv_bfloat16* __restrict__ Xb, int64_t ldxb, int Ep) {
  if (seed_dev) seed += *seed_dev;
  // one warp per packed row
  int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= N) return;
  int lane = threadIdx.x & 31;
  int b = row_b[row], t = row_t[row];
  int ov = tok_override ? tok_override[row] : -1;
  float* dst = X ? X + row * ldx : nullptr;
  __nv_bfloat16* dstb = Xb ? Xb + row * ldxb : nullptr;
  const float* src;
  float pp = 0.f;
  if (ov < 0 && has_feat && t == 0) {
    src = features + (int64_t)b * feat_ld;
  } else {
    int64_t tok = ov >= 0 ? (int64_t)ov : captions[(int64_t)b * cap_ld + (t - has_feat)];
    src = table + tok * E;
    pp = ov >= 0 ? 0.f : p;   // fed-back embeddings are not dropped out (model.py:184)
  }
  for (int c = lane; c < Ep; c += 32) {
    float v = c < E ? src[c] * sn::dropout_scale(seed, (uint32_t)row, (uint32_t)c, pp, inv_keep) : 0.f;
    if (dst && c < E) dst[c] = v;
    if (dstb) dstb[c] = __float2bfloat16(v);     // columns E..Ep are the zero K-padding of the TMA operand
  }
}

__global__ void gather_pack_bwd_kernel(const int64_t* __restrict__ captions, int64_t cap_ld,
                                       float* __restrict__ dtable, int E, float* __restrict__ dfeatures,
                                       int64_t feat_ld, int has_feat, const int32_t* __restrict__ row_b,
                                       const int32_t* __restrict__ row_t,
                                       const int32_t* __restrict__ tok_override, int64_t N,
                                       const float* __restrict__ dX, int64_t ldx, float p, float inv_keep,
                                       uint64_t seed, const uint64_t* __restrict__ seed_dev) {
  if (seed_dev) seed += *seed_dev;
  int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= N) return;
  int lane = threadIdx.x & 31;
  int b = row_b[row], t = row_t[row];
  int ov = tok_override ? tok_override[row] : -1;
  const float* src = dX + row * ldx;
  if (ov < 0 && has_feat && t == 0) {
    if (dfeatures) {
      float* dst = dfeatures + (int64_t)b * feat_ld;
      for (int c = lane; c < E; c += 32) dst[c] = src[c];
    }
    return;
  }
  // token rows: embed_*_kernel below
}

// token of packed row i (-1: the image-feature row)
__device__ __forceinline__ int64_t packed_token(int64_t i, const int64_t* __restrict__ captions, int64_t cap_ld,
                                                int has_feat, const int32_t* __restrict__ row_b,
                                                const int32_t* __restrict__ row_t,
                                                const int32_t* __restrict__ tok_override) {
  int ov = tok_override ? tok_override[i] : -1;
  if (ov >= 0) return ov;
  int t = row_t[i];
  if (has_feat && t == 0) return -1;
  return captions[(int64_t)row_b[i] * cap_ld + (t - has_feat)];
}

// Embedding gradient without float atomics, so that the sum (and the Adam step behind it) is the same from run to run.
// The token rows are grouped by token with a counting sort, each group is put in row order, and each group is summed
// in fixed chunks of EB_CHUNK rows; a group longer than one chunk adds its chunk sums in chunk order.  Every kernel is
// parallel over rows, slots or tokens: the cost grows with N (ordering a group of s rows costs s^2 compares, which
// for the <start> / <end> groups of B rows each is B^2).
constexpr int EB_CHUNK = 32;  // rows summed by one warp
constexpr int EB_K = 16;      // columns per lane and pass: 512 per pass

// token of every row (-1: image-feature row) and rows per token (integer atomics: the counts are exact)
__global__ void embed_count_kernel(const int64_t* __restrict__ captions, int64_t cap_ld, int has_feat,
                                   const int32_t* __restrict__ row_b, const int32_t* __restrict__ row_t,
                                   const int32_t* __restrict__ tok_override, int64_t N, int32_t* __restrict__ tok32,
                                   int32_t* __restrict__ cnt) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= N) return;
  const int64_t t = packed_token(r, captions, cap_ld, has_feat, row_b, row_t, tok_override);
  tok32[r] = (int32_t)t;
  if (t >= 0) atomicAdd(cnt + t, 1);
}

// one CTA of 1024: start = exclusive scan of cnt (start[V] = token rows), cursor = start, cstart = exclusive scan of the
// chunk count of every group longer than one chunk
__global__ void __launch_bounds__(1024) embed_scan_kernel(const int32_t* __restrict__ cnt, int64_t V,
                                                          int32_t* __restrict__ start, int32_t* __restrict__ cursor,
                                                          int32_t* __restrict__ cstart) {
  __shared__ int32_t s1[1024], s2[1024];
  const int tid = threadIdx.x;
  const int64_t per = (V + 1023) / 1024, lo = tid * per, hi = lo + per < V ? lo + per : V;
  int32_t a = 0, c = 0;
  for (int64_t v = lo; v < hi; ++v) {
    const int32_t n = cnt[v];
    a += n;
    c += n > EB_CHUNK ? (n + EB_CHUNK - 1) / EB_CHUNK : 0;
  }
  s1[tid] = a; s2[tid] = c;
  __syncthreads();
  for (int off = 1; off < 1024; off <<= 1) {       // Hillis-Steele inclusive scan
    const int32_t x = tid >= off ? s1[tid - off] : 0, y = tid >= off ? s2[tid - off] : 0;
    __syncthreads();
    s1[tid] += x; s2[tid] += y;
    __syncthreads();
  }
  a = s1[tid] - a; c = s2[tid] - c;
  for (int64_t v = lo; v < hi; ++v) {
    const int32_t n = cnt[v];
    start[v] = a; cursor[v] = a; cstart[v] = c;
    a += n;
    c += n > EB_CHUNK ? (n + EB_CHUNK - 1) / EB_CHUNK : 0;
  }
  if (tid == 1023) start[V] = s1[1023];
}

// rows into their token's group (order inside a group still arbitrary)
__global__ void embed_place_kernel(const int32_t* __restrict__ tok32, int64_t N, int32_t* __restrict__ cursor,
                                   int32_t* __restrict__ perm) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= N) return;
  const int32_t t = tok32[r];
  if (t >= 0) perm[atomicAdd(cursor + t, 1)] = (int32_t)r;
}

// row order inside every group: a row's rank is the number of smaller row indices in its group
__global__ void embed_order_kernel(const int32_t* __restrict__ tok32, const int32_t* __restrict__ start,
                                   const int32_t* __restrict__ perm, int64_t N, int64_t V,
                                   int32_t* __restrict__ sorted) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= start[V]) return;
  const int32_t r = perm[i], t = tok32[r], s = start[t], e = start[t + 1];
  int32_t rank = 0;
  for (int32_t j = s; j < e; ++j) rank += perm[j] < r;
  sorted[s + rank] = r;
}

// one warp per chunk of a group: the chunk's rows in row order; a group of one chunk goes straight to dtable
__global__ void embed_chunk_kernel(const int32_t* __restrict__ tok32, const int32_t* __restrict__ start,
                                   const int32_t* __restrict__ cstart, const int32_t* __restrict__ sorted, int64_t V,
                                   const int32_t* __restrict__ tok_override, const float* __restrict__ dX, int64_t ldx,
                                   int E, float p, float inv_keep, uint64_t seed, const uint64_t* __restrict__ seed_dev,
                                   float* __restrict__ dtable, float* __restrict__ part) {
  if (seed_dev) seed += *seed_dev;
  const int64_t i = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (i >= start[V]) return;
  const int lane = threadIdx.x & 31;
  const int32_t t = tok32[sorted[i]], s = start[t], e = start[t + 1];
  if ((i - s) % EB_CHUNK) return;
  const int32_t n = (int32_t)(e - i < EB_CHUNK ? e - i : EB_CHUNK);
  const int32_t my = lane < n ? sorted[i + lane] : 0;
  float* dst = e - s <= EB_CHUNK ? dtable + (int64_t)t * E : part + (int64_t)(cstart[t] + (i - s) / EB_CHUNK) * E;
  for (int c0 = 0; c0 < E; c0 += 32 * EB_K) {
    float acc[EB_K];
#pragma unroll
    for (int k = 0; k < EB_K; ++k) acc[k] = 0.f;
    for (int q = 0; q < n; ++q) {
      const int64_t j = __shfl_sync(0xffffffffu, my, q);
      const float pp = (tok_override && tok_override[j] >= 0) ? 0.f : p;   // fed-back embeddings: no dropout
      const float* src = dX + j * ldx;
#pragma unroll
      for (int k = 0; k < EB_K; ++k) {
        const int c = c0 + k * 32 + lane;
        if (c < E) {
          const float sc = sn::dropout_scale(seed, (uint32_t)j, (uint32_t)c, pp, inv_keep);
          if (sc != 0.f) acc[k] += src[c] * sc;
        }
      }
    }
#pragma unroll
    for (int k = 0; k < EB_K; ++k) {
      const int c = c0 + k * 32 + lane;
      if (c < E) {
        if (e - s <= EB_CHUNK) dst[c] += acc[k];
        else dst[c] = acc[k];
      }
    }
  }
}

// The same chunk sums as embed_chunk_kernel, bit for bit, with the latency of a chunk cut: one CTA per chunk and one
// thread per column (blockDim.x >= E, a multiple of 32), the chunk's row ids and dropout rates staged in shared memory,
// and the rows loaded EBW_BATCH at a time before they are added in row order.  A row with scale 0 is loaded but not
// added, exactly as the warp kernel skips it (acc + 0 would turn an accumulated -0 into +0); the product-sum is the FFMA
// the warp kernel compiles to.  The warp kernel pays one dependent load round per row: ~70 us at configs[1], where
// the <start> token's 96 rows make three chunks of 32 (B200, profiles/README.md).
constexpr int EBW_BATCH = 16;
__global__ void __launch_bounds__(512) embed_chunk_wide_kernel(
    const int32_t* __restrict__ tok32, const int32_t* __restrict__ start, const int32_t* __restrict__ cstart,
    const int32_t* __restrict__ sorted, int64_t V, const int32_t* __restrict__ tok_override,
    const float* __restrict__ dX, int64_t ldx, int E, float p, float inv_keep, uint64_t seed,
    const uint64_t* __restrict__ seed_dev, float* __restrict__ dtable, float* __restrict__ part) {
  __shared__ int32_t rows[EB_CHUNK];
  __shared__ float rate[EB_CHUNK];
  const int64_t i = blockIdx.x;
  if (i >= start[V]) return;
  const int32_t t = tok32[sorted[i]], s = start[t], e = start[t + 1];
  if ((i - s) % EB_CHUNK) return;
  if (seed_dev) seed += *seed_dev;
  const int32_t n = (int32_t)(e - i < EB_CHUNK ? e - i : EB_CHUNK);
  if (threadIdx.x < n) {
    const int32_t j = sorted[i + threadIdx.x];
    rows[threadIdx.x] = j;
    rate[threadIdx.x] = (tok_override && tok_override[j] >= 0) ? 0.f : p;   // fed-back embeddings: no dropout
  }
  __syncthreads();
  const int c = threadIdx.x;
  if (c >= E) return;
  float acc = 0.f;
  for (int q0 = 0; q0 < n; q0 += EBW_BATCH) {
    float x[EBW_BATCH], sc[EBW_BATCH];
#pragma unroll
    for (int u = 0; u < EBW_BATCH; ++u) {
      const int q = q0 + u;
      x[u] = 0.f; sc[u] = 0.f;
      if (q < n) {
        const int64_t j = rows[q];
        x[u] = dX[j * ldx + c];
        sc[u] = sn::dropout_scale(seed, (uint32_t)j, (uint32_t)c, rate[q], inv_keep);
      }
    }
#pragma unroll
    for (int u = 0; u < EBW_BATCH; ++u)
      if (sc[u] != 0.f) acc = __fmaf_rn(x[u], sc[u], acc);
  }
  if (e - s <= EB_CHUNK) dtable[(int64_t)t * E + c] += acc;
  else part[(int64_t)(cstart[t] + (i - s) / EB_CHUNK) * E + c] = acc;
}

// one warp per token whose group has several chunks: chunk sums in chunk order
__global__ void embed_combine_kernel(const int32_t* __restrict__ cnt, const int32_t* __restrict__ cstart, int64_t V,
                                     int E, const float* __restrict__ part, float* __restrict__ dtable) {
  const int64_t t = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (t >= V || cnt[t] <= EB_CHUNK) return;
  const int lane = threadIdx.x & 31;
  const int32_t nq = (cnt[t] + EB_CHUNK - 1) / EB_CHUNK;
  const float* src = part + (int64_t)cstart[t] * E;
  for (int c = lane; c < E; c += 32) {
    float a = 0.f;
    for (int32_t q = 0; q < nq; ++q) a += src[(int64_t)q * E + c];
    dtable[t * E + c] += a;
  }
}

// ------------------------------------------------------------------------------------------
// K5: one CTA per row; the row (V floats) is staged in shared memory so HBM sees one read of the
// logits and (optionally) one write of the gradient.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) softmax_nll_kernel(const float* __restrict__ logits, int64_t V, int64_t ld,
                                                          const int64_t* __restrict__ targets,
                                                          float* __restrict__ row_loss, float* dlogits, int64_t ldd,
                                                          float grad_scale, const float* __restrict__ row_weight,
                                                          int64_t* __restrict__ argmax,
                                                          int32_t* __restrict__ top5hit, int use_smem,
                                                          __nv_bfloat16* __restrict__ dlb, int64_t lddb) {
  extern __shared__ float srow[];
  __shared__ float red_v[8];
  __shared__ int red_i[8];
  __shared__ float bc_f[2];
  __shared__ int bc_i;
  const int64_t row = blockIdx.x;
  const float* src = logits + row * ld;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

  // pass 1: max + first arg-max
  float mx = -INFINITY;
  int mi = 0x7fffffff;
  for (int64_t c = tid; c < V; c += 256) {
    float v = src[c];
    if (use_smem) srow[c] = v;
    if (v > mx) { mx = v; mi = (int)c; }   // strictly greater keeps the lowest index per thread
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    float ov = __shfl_xor_sync(0xffffffffu, mx, o);
    int oi = __shfl_xor_sync(0xffffffffu, mi, o);
    if (ov > mx || (ov == mx && oi < mi)) { mx = ov; mi = oi; }
  }
  if (lane == 0) { red_v[warp] = mx; red_i[warp] = mi; }
  __syncthreads();
  if (tid == 0) {
    float bm = red_v[0]; int bi = red_i[0];
    for (int w = 1; w < 8; ++w)
      if (red_v[w] > bm || (red_v[w] == bm && red_i[w] < bi)) { bm = red_v[w]; bi = red_i[w]; }
    bc_f[0] = bm; bc_i = bi;
  }
  __syncthreads();
  mx = bc_f[0];
  if (tid == 0 && argmax) argmax[row] = bc_i;
  if (!targets) return;

  const float* rd = use_smem ? srow : src;
  const int64_t tgt = targets[row];
  const float tv = rd[tgt];
  // pass 2: sum exp, count of logits strictly above the target's
  float se = 0.f;
  int above = 0;
  for (int64_t c = tid; c < V; c += 256) {
    float v = rd[c];
    se += expf(v - mx);
    above += (v > tv);
  }
  se = sn::warp_sum(se);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) above += __shfl_xor_sync(0xffffffffu, above, o);
  __syncthreads();
  if (lane == 0) { red_v[warp] = se; red_i[warp] = above; }
  __syncthreads();
  if (tid == 0) {
    float s = 0.f; int a = 0;
    for (int w = 0; w < 8; ++w) { s += red_v[w]; a += red_i[w]; }
    float lse = mx + logf(s);
    bc_f[1] = lse;
    if (row_loss) row_loss[row] = lse - tv;
    if (top5hit) top5hit[row] = a < 5 ? 1 : 0;
  }
  __syncthreads();
  if (dlogits || dlb) {
    const float lse = bc_f[1];
    const float gs = row_weight ? grad_scale * row_weight[row] : grad_scale;
    float* dst = dlogits ? dlogits + row * ldd : nullptr;
    __nv_bfloat16* dstb = dlb ? dlb + row * lddb : nullptr;
    for (int64_t c = tid; c < V; c += 256) {
      float pr = expf(rd[c] - lse);
      float gr = (pr - (c == tgt ? 1.f : 0.f)) * gs;
      if (dst) dst[c] = gr;
      if (dstb) dstb[c] = __float2bfloat16(gr);
    }
    if (dstb) for (int64_t c = V + tid; c < lddb; c += 256) dstb[c] = __float2bfloat16(0.f);
  }
}

__global__ void __launch_bounds__(1024) reduce_sum_kernel(const float* __restrict__ x, int64_t N, float scale,
                                                           const float* __restrict__ w, float* out, int accumulate) {
  __shared__ double part[32];
  double s = 0.0;
  if (w)
    for (int64_t i = threadIdx.x; i < N; i += 1024) s += (double)x[i] * (double)w[i];
  else
    for (int64_t i = threadIdx.x; i < N; i += 1024) s += (double)x[i];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int w = 0; w < 32; ++w) t += part[w];
    float r = (float)(t * (double)scale);
    *out = accumulate ? *out + r : r;
  }
}

// ------------------------------------------------------------------------------------------
// K7: clamp + Adam, torch.optim.Adam op order (see sn100.h)
// ------------------------------------------------------------------------------------------
struct AdamRanges {
  // passed BY VALUE to every optimizer / exchange kernel: kept under the classic 4 KB kernel-parameter limit (28 bytes per
  // range) -- with 36-byte entries the 128-range struct was 5.5 KB and the configs[1] step got 17 us slower (8 launches)
  static constexpr int MAX = 128;
  int64_t off[MAX];
  int32_t len[MAX];
  float step_size[MAX], bc2_sqrt[MAX];
  int step_idx[MAX];              // device-step mode: index into steps_dev
  int32_t chunk_start[MAX + 1];   // prefix of per-range chunk counts
  int n;
};
static_assert(sizeof(AdamRanges) <= 3700, "AdamRanges must leave room for the other kernel parameters below 4 KB");

// device-step mode: bump the step counter of every range's parameter and derive the bias-corrected
// coefficients exactly like torch.optim.Adam does on the host (double precision)
__global__ void adam_prepare_kernel(AdamRanges R, int32_t* __restrict__ steps, const float* __restrict__ lr,
                                    float* __restrict__ coef, float beta1, float beta2) {
  int r = threadIdx.x;
  if (r >= R.n) return;
  int st = steps[R.step_idx[r]] + 1;
  steps[R.step_idx[r]] = st;
  double bc1 = 1.0 - pow((double)beta1, (double)st);
  double bc2 = 1.0 - pow((double)beta2, (double)st);
  // slot = the parameter's step index, not the position in this call: calls that run concurrently on different
  // streams (bucketed early steps) cover disjoint parameters and therefore never share a slot
  coef[2 * R.step_idx[r]] = (float)((double)(*lr) / bc1);
  coef[2 * R.step_idx[r] + 1] = (float)sqrt(bc2);
}
constexpr int ADAM_CHUNK = 4096;   // elements per CTA-iteration
constexpr int64_t ADAM_MAX_LEN = (1LL << 31) - 2 * ADAM_CHUNK;      // a range's length is an int32 in AdamRanges

__global__ void __launch_bounds__(256) adam_clamp_kernel(float* __restrict__ p, float* __restrict__ g,
                                                         float* __restrict__ m, float* __restrict__ v,
                                                         AdamRanges R, const float* __restrict__ coef, float beta1,
                                                         float beta2, float eps, float clip) {
  const int64_t total_chunks = R.chunk_start[R.n];
  for (int64_t ch = blockIdx.x; ch < total_chunks; ch += gridDim.x) {
    int r = 0;
    while (ch >= R.chunk_start[r + 1]) ++r;
    const int64_t base = R.off[r] + (ch - R.chunk_start[r]) * ADAM_CHUNK;
    const int64_t end = R.off[r] + R.len[r];
    const float ss = coef ? coef[2 * R.step_idx[r]] : R.step_size[r], bc = coef ? coef[2 * R.step_idx[r] + 1] : R.bc2_sqrt[r];
    const int64_t lim = base + ADAM_CHUNK < end ? base + ADAM_CHUNK : end;
    if ((base & 3) == 0 && lim - base == ADAM_CHUNK) {
      // full, 16-byte aligned chunk: 128-bit loads/stores, 4 independent elements per thread per pass
#pragma unroll
      for (int it = 0; it < ADAM_CHUNK / (256 * 4); ++it) {
        const int64_t i = base + (int64_t)(it * 256 + threadIdx.x) * 4;
        float4 g4 = *reinterpret_cast<const float4*>(g + i);
        float4 m4 = *reinterpret_cast<const float4*>(m + i);
        float4 v4 = *reinterpret_cast<const float4*>(v + i);
        float4 p4 = *reinterpret_cast<const float4*>(p + i);
        float* gp = &g4.x; float* mp = &m4.x; float* vp = &v4.x; float* pp = &p4.x;
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          float gi = gp[e];
          if (clip > 0.f) gi = fminf(fmaxf(gi, -clip), clip);
          gp[e] = gi;
          float mi = mp[e] + (1.f - beta1) * (gi - mp[e]);
          float vi = vp[e] * beta2 + (1.f - beta2) * gi * gi;
          float denom = sqrtf(vi) / bc + eps;
          pp[e] = pp[e] - ss * (mi / denom);
          mp[e] = mi; vp[e] = vi;
        }
        if (clip > 0.f) *reinterpret_cast<float4*>(g + i) = g4;       // clamp_ is in place (utils.py:60)
        *reinterpret_cast<float4*>(m + i) = m4;
        *reinterpret_cast<float4*>(v + i) = v4;
        *reinterpret_cast<float4*>(p + i) = p4;
      }
      continue;
    }
    for (int64_t i = base + threadIdx.x; i < lim; i += 256) {
      float gi = g[i];
      if (clip > 0.f) { gi = fminf(fmaxf(gi, -clip), clip); g[i] = gi; }   // clamp_ is in place (utils.py:60)
      float mi = m[i], vi = v[i];
      mi = mi + (1.f - beta1) * (gi - mi);
      vi = vi * beta2 + (1.f - beta2) * gi * gi;
      float denom = sqrtf(vi) / bc + eps;
      p[i] = p[i] - ss * (mi / denom);
      m[i] = mi; v[i] = vi;
    }
  }
}

// ------------------------------------------------------------------------------------------------------
// Data-parallel exchange fused with the optimizer (K9+K7): reduce-scatter of the gradients over NVLink peer
// memory -> clamp + Adam on this rank's shard -> all-gather of the updated parameters by peer stores, in ONE
// kernel and with no NCCL call.  Every rank runs the same kernel on its own GPU; chunk c (4096 elements of the
// concatenated active ranges) belongs to rank c % world.  Cross-GPU ordering uses two epoch flags per peer in
// a small "pad" that lives in every rank's memory (arrive: my gradients are final; done: I have read every
// gradient I need and my parameter stores have landed).
// ------------------------------------------------------------------------------------------------------
struct DpPeers {
  float* grad[8];
  float* param[8];
  int* pad[8];
  int world, rank;
  // push form: every rank's receive buffer (world slots of `slot_elems` elements each: slot q of rank o holds rank q's
  // gradients of the chunks o owns, chunk `aid` at element (aid / world) * ADAM_CHUNK), element size 4 (fp32) or 2 (bf16)
  void* recv[8];
  int64_t slot_elems;
  int* wait_pad[4];     // my pads of the push buckets this call consumes (ARRIVE flags written by the peers' pushes)
  int n_wait;
};
constexpr int PAD_ARRIVE = 0, PAD_DONE = 8, PAD_COUNTER = 16, PAD_EPOCH = 17, PAD_DONE_COUNTER = 18;

__device__ __forceinline__ int ld_acquire_sys(const int* p) {
  int v;
  asm volatile("ld.acquire.sys.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_sys(int* p, int v) {
  asm volatile("st.release.sys.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// ---- push form, part 1: send my gradients of the chunks I do NOT own to their owners (posted NVLink stores: nothing
// waits here), then raise my ARRIVE flag in every peer's pad.  Launched on the stream that produced the gradients as
// soon as a bucket is final, so the transfer runs under the rest of the backward.
// Fat CTAs (DP_SUB groups of 256 threads, one chunk per group and iteration, at most one CTA per SM): the system-scope
// fence that closes a CTA costs microseconds once remote stores are in flight and the fences of the CTAs of one SM do
// not overlap -- one per SM instead of one per 256 threads took the kernel from ~17 us + data to ~6 us + data.
constexpr int DP_SUB = 4;
template <typename TT>
__global__ void __launch_bounds__(256 * DP_SUB) dp_push_kernel(DpPeers P, AdamRanges R, const float* __restrict__ g) {
  const int W = P.world;
  __shared__ int s_last;
  int* mypad = P.pad[P.rank];
  const int64_t total_chunks = R.chunk_start[R.n];
  const int sub = threadIdx.x >> 8, tid = threadIdx.x & 255;
  for (int64_t ch = (int64_t)blockIdx.x * DP_SUB + sub; ch < total_chunks; ch += (int64_t)gridDim.x * DP_SUB) {
    int r = 0;
    while (ch >= R.chunk_start[r + 1]) ++r;
    const int64_t aid = R.off[r] / ADAM_CHUNK + (ch - R.chunk_start[r]);
    const int owner = (int)(aid % W);
    if (owner == P.rank) continue;
    const int64_t end = R.off[r] + R.len[r];
    const int64_t base = aid * ADAM_CHUNK > R.off[r] ? aid * ADAM_CHUNK : R.off[r];
    const int64_t lim = (aid + 1) * ADAM_CHUNK < end ? (aid + 1) * ADAM_CHUNK : end;
    TT* dst = reinterpret_cast<TT*>(P.recv[owner]) + (int64_t)P.rank * P.slot_elems + (aid / W) * ADAM_CHUNK - aid * ADAM_CHUNK;
    if ((base & 3) == 0 && lim - base == ADAM_CHUNK) {
      float4 t[ADAM_CHUNK / 1024];
#pragma unroll
      for (int u = 0; u < ADAM_CHUNK / 1024; ++u)
        t[u] = __ldcg(reinterpret_cast<const float4*>(g + base + (int64_t)(u * 256 + tid) * 4));
#pragma unroll
      for (int u = 0; u < ADAM_CHUNK / 1024; ++u) {
        const int64_t i = base + (int64_t)(u * 256 + tid) * 4;
        if constexpr (sizeof(TT) == 4) {
          *reinterpret_cast<float4*>(dst + i) = t[u];
        } else {
          __nv_bfloat162 lo = __floats2bfloat162_rn(t[u].x, t[u].y), hi = __floats2bfloat162_rn(t[u].z, t[u].w);
          uint2 pk;
          pk.x = *reinterpret_cast<uint32_t*>(&lo); pk.y = *reinterpret_cast<uint32_t*>(&hi);
          *reinterpret_cast<uint2*>(dst + i) = pk;
        }
      }
      continue;
    }
    for (int64_t i = base + tid; i < lim; i += 256) {
      if constexpr (sizeof(TT) == 4) dst[i] = g[i]; else dst[i] = __float2bfloat16_rn(g[i]);
    }
  }
  // my stores are on their way: one system fence per block (cumulative over the block's stores through the barrier),
  // count blocks, the last one tells every peer
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence_system();
    s_last = (atomicAdd(mypad + PAD_COUNTER, 1) == (int)gridDim.x - 1);
  }
  __syncthreads();
  if (s_last) {
    if (threadIdx.x == 0) {
      __threadfence_system();
      const int e = mypad[PAD_EPOCH] + 1;
      for (int q = 0; q < W; ++q) st_release_sys(P.pad[q] + PAD_ARRIVE + P.rank, e);
      mypad[PAD_COUNTER] = 0;
    }
  }
}

template <int W>      // world size as a template parameter: the W peer loads / stores of an element are all in flight
__global__ void __launch_bounds__(256) dp_adam_fused_kernel(DpPeers P, AdamRanges R, const float* __restrict__ coef,
                                                            float* __restrict__ m, float* __restrict__ v, float beta1,
                                                            float beta2, float eps, float clip, int dbg) {
  if (dbg) {        // timing experiments only (SN_DP_DEBUG): bit 0 = local gradient reads only, bit 1 = local stores only
    for (int q = 0; q < P.world; ++q) {
      if (dbg & 1) P.grad[q] = P.grad[P.rank];
      if (dbg & 2) P.param[q] = P.param[P.rank];
    }
  }
  __shared__ int s_epoch, s_last;
  int* mypad = P.pad[P.rank];
  if (threadIdx.x == 0) s_epoch = mypad[PAD_EPOCH] + 1;
  __syncthreads();
  const int e = s_epoch;
  // 1. my gradients are final (stream order): tell every peer; 2. wait until every peer said the same
  if (blockIdx.x == 0 && threadIdx.x < P.world) st_release_sys(P.pad[threadIdx.x] + PAD_ARRIVE + P.rank, e);
  if (threadIdx.x < P.world) { while (ld_acquire_sys(mypad + PAD_ARRIVE + threadIdx.x) < e) { } }
  __syncthreads();
  // 3. my chunks: reduce over the peers (fixed rank order), clamp, Adam, store the new parameters everywhere.
  // Ownership is a function of the ABSOLUTE arena offset only -- element i belongs to rank (i / ADAM_CHUNK) % world --
  // so it does not move when the set of active ranges changes between calls (early / late exchange, accumulation,
  // only= / skip=): the Adam moments of an element always live on the same rank.  Chunks are therefore cut on the
  // absolute ADAM_CHUNK grid and clipped to their range; a slot of W consecutive chunks holds (about) one owned chunk.
  const int64_t total_chunks = R.chunk_start[R.n];
  const int64_t nslots = (total_chunks + W - 1) / W;
  for (int64_t slot = blockIdx.x; slot < nslots; slot += gridDim.x)
  for (int j = 0; j < W; ++j) {
    const int64_t ch = slot * W + j;
    if (ch >= total_chunks) break;
    int r = 0;
    while (ch >= R.chunk_start[r + 1]) ++r;
    const int64_t aid = R.off[r] / ADAM_CHUNK + (ch - R.chunk_start[r]);      // absolute chunk id
    if ((int)(aid % W) != P.rank) continue;
    const int64_t end = R.off[r] + R.len[r];
    const int64_t base = aid * ADAM_CHUNK > R.off[r] ? aid * ADAM_CHUNK : R.off[r];
    const int64_t lim = (aid + 1) * ADAM_CHUNK < end ? (aid + 1) * ADAM_CHUNK : end;
    const float ss = coef[2 * R.step_idx[r]], bc = coef[2 * R.step_idx[r] + 1];
    if ((base & 3) == 0 && lim - base == ADAM_CHUNK) {
      // NIT iterations at a time with ALL their loads issued up front: the peer loads cross NVLink (~2 us each), so the
      // number of them in flight per thread, not the instruction count, sets the pace
      constexpr int NIT = W <= 4 ? 4 : 2;
#pragma unroll
      for (int it0 = 0; it0 < ADAM_CHUNK / (256 * 4); it0 += NIT) {
        float4 t[NIT][W], m4[NIT], v4[NIT], p4[NIT];
#pragma unroll
        for (int u = 0; u < NIT; ++u) {
          const int64_t i = base + (int64_t)((it0 + u) * 256 + threadIdx.x) * 4;
#pragma unroll
          for (int q = 0; q < W; ++q) t[u][q] = __ldcg(reinterpret_cast<const float4*>(P.grad[q] + i));
        }
#pragma unroll
        for (int u = 0; u < NIT; ++u) {
          const int64_t i = base + (int64_t)((it0 + u) * 256 + threadIdx.x) * 4;
          m4[u] = *reinterpret_cast<const float4*>(m + i);
          v4[u] = *reinterpret_cast<const float4*>(v + i);
          p4[u] = *reinterpret_cast<const float4*>(P.param[P.rank] + i);
        }
#pragma unroll
        for (int u = 0; u < NIT; ++u) {
          const int64_t i = base + (int64_t)((it0 + u) * 256 + threadIdx.x) * 4;
          float4 g4 = t[u][0];
#pragma unroll
          for (int q = 1; q < W; ++q) { g4.x += t[u][q].x; g4.y += t[u][q].y; g4.z += t[u][q].z; g4.w += t[u][q].w; }
          float* gp = &g4.x; float* mp = &m4[u].x; float* vp = &v4[u].x; float* pp = &p4[u].x;
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            float gi = gp[k];
            if (clip > 0.f) gi = fminf(fmaxf(gi, -clip), clip);
            const float mi = mp[k] + (1.f - beta1) * (gi - mp[k]);
            const float vi = vp[k] * beta2 + (1.f - beta2) * gi * gi;
            pp[k] = pp[k] - ss * (mi / (sqrtf(vi) / bc + eps));
            mp[k] = mi; vp[k] = vi;
          }
          *reinterpret_cast<float4*>(m + i) = m4[u];
          *reinterpret_cast<float4*>(v + i) = v4[u];
#pragma unroll
          for (int q = 0; q < W; ++q) *reinterpret_cast<float4*>(P.param[q] + i) = p4[u];
        }
      }
      continue;
    }
    for (int64_t i = base + threadIdx.x; i < lim; i += 256) {
      float gi = __ldcg(P.grad[0] + i);
#pragma unroll
      for (int q = 1; q < W; ++q) gi += __ldcg(P.grad[q] + i);
      if (clip > 0.f) gi = fminf(fmaxf(gi, -clip), clip);
      const float mi = m[i] + (1.f - beta1) * (gi - m[i]);
      const float vi = v[i] * beta2 + (1.f - beta2) * gi * gi;
      const float pn = P.param[P.rank][i] - ss * (mi / (sqrtf(vi) / bc + eps));
      m[i] = mi; v[i] = vi;
#pragma unroll
      for (int q = 0; q < W; ++q) P.param[q][i] = pn;
    }
  }
  // 4. all my reads are done and my stores are on their way: one system fence per block (cumulative over the block's
  // accesses through the barrier), count blocks, last block runs the exit barrier
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence_system();
    s_last = (atomicAdd(mypad + PAD_DONE_COUNTER, 1) == (int)gridDim.x - 1);
  }
  __syncthreads();
  if (s_last) {
    if (threadIdx.x == 0) __threadfence_system();
    __syncthreads();
    if (threadIdx.x < P.world) {
      st_release_sys(P.pad[threadIdx.x] + PAD_DONE + P.rank, e);
      while (ld_acquire_sys(mypad + PAD_DONE + threadIdx.x) < e) { }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      mypad[PAD_DONE_COUNTER] = 0; mypad[PAD_EPOCH] = e;
    }
  }
}

// ---- push form, part 2: the peers' gradients of my chunks are in my receive buffer (dp_push_kernel).  Wait for their
// ARRIVE flags (local polls), reduce own fp32 gradient + the received ones in rank order, clamp, Adam on the owned
// chunks, store the new parameters to every rank, exit barrier.  Written like adam_clamp_kernel (one chunk per CTA
// iteration, few registers, many CTAs per SM) -- the per-CTA flag poll and exit fence hide under the neighbours' loads.
// R.chunk_start counts OWNED chunks only (host), so the CTAs share the owned chunks evenly for every world size.
constexpr int DP_RSUB = 2;
template <int W, typename TT>
__global__ void __launch_bounds__(256 * DP_RSUB) dp_recv_adam_kernel(DpPeers P, AdamRanges R, const float* __restrict__ coef,
                                                           const float* __restrict__ g, const TT* __restrict__ recv,
                                                           const float* p_loc, float* __restrict__ m, float* __restrict__ v, float beta1,
                                                           float beta2, float eps, float clip) {
  __shared__ int s_epoch, s_last;
  const int rank = P.rank;
  int* mypad = P.wait_pad[0];
  if (threadIdx.x == 0) s_epoch = mypad[PAD_EPOCH] + 1;
  if (threadIdx.x < W * P.n_wait) {
    const int* wp = P.wait_pad[threadIdx.x / W];
    const int q = threadIdx.x % W;
    if (q != rank) { const int we = wp[PAD_EPOCH] + 1; while (ld_acquire_sys(wp + PAD_ARRIVE + q) < we) { } }
  }
  __syncthreads();
  const int e = s_epoch;
  const int64_t total_chunks = R.chunk_start[R.n];
  const int sub = threadIdx.x >> 8, tid = threadIdx.x & 255;
  for (int64_t ch = (int64_t)blockIdx.x * DP_RSUB + sub; ch < total_chunks; ch += (int64_t)gridDim.x * DP_RSUB) {
    int r = 0;
    while (ch >= R.chunk_start[r + 1]) ++r;
    const int64_t a0 = R.off[r] / ADAM_CHUNK;
    const int64_t aid = a0 + ((rank - a0) % W + W) % W + (ch - R.chunk_start[r]) * W;     // my (ch - start)-th chunk of range r
    const int64_t end = R.off[r] + R.len[r];
    const int64_t base = aid * ADAM_CHUNK > R.off[r] ? aid * ADAM_CHUNK : R.off[r];
    const int64_t lim = (aid + 1) * ADAM_CHUNK < end ? (aid + 1) * ADAM_CHUNK : end;
    const float ss = coef[2 * R.step_idx[r]], bc = coef[2 * R.step_idx[r] + 1];
    const int64_t rbase = (aid / W) * ADAM_CHUNK - aid * ADAM_CHUNK;      // arena index -> index in a receive slot
    if ((base & 3) == 0 && lim - base == ADAM_CHUNK) {
#pragma unroll
      for (int it = 0; it < ADAM_CHUNK / (256 * 4); ++it) {
        const int64_t i = base + (int64_t)(it * 256 + tid) * 4;
        float4 t[W];
#pragma unroll
        for (int q = 0; q < W; ++q) {
          if (q == rank) {
            t[q] = __ldcg(reinterpret_cast<const float4*>(g + i));
          } else if constexpr (sizeof(TT) == 4) {
            t[q] = __ldcg(reinterpret_cast<const float4*>(recv + q * P.slot_elems + rbase + i));
          } else {
            const uint2 pk = __ldcg(reinterpret_cast<const uint2*>(recv + q * P.slot_elems + rbase + i));
            const float2 lo = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&pk.x));
            const float2 hi = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&pk.y));
            t[q] = make_float4(lo.x, lo.y, hi.x, hi.y);
          }
        }
        float4 m4 = *reinterpret_cast<const float4*>(m + i);
        float4 v4 = *reinterpret_cast<const float4*>(v + i);
        float4 p4 = *reinterpret_cast<const float4*>(p_loc + i);
        float4 g4 = t[0];
#pragma unroll
        for (int q = 1; q < W; ++q) { g4.x += t[q].x; g4.y += t[q].y; g4.z += t[q].z; g4.w += t[q].w; }
        float* gp = &g4.x; float* mp = &m4.x; float* vp = &v4.x; float* pp = &p4.x;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          float gi = gp[k];
          if (clip > 0.f) gi = fminf(fmaxf(gi, -clip), clip);
          const float mi = mp[k] + (1.f - beta1) * (gi - mp[k]);
          const float vi = vp[k] * beta2 + (1.f - beta2) * gi * gi;
          pp[k] = pp[k] - ss * (mi / (sqrtf(vi) / bc + eps));
          mp[k] = mi; vp[k] = vi;
        }
        *reinterpret_cast<float4*>(m + i) = m4;
        *reinterpret_cast<float4*>(v + i) = v4;
#pragma unroll
        for (int q = 0; q < W; ++q) *reinterpret_cast<float4*>(P.param[q] + i) = p4;
      }
      continue;
    }
    for (int64_t i = base + tid; i < lim; i += 256) {
      float gi = 0.f;
#pragma unroll
      for (int q = 0; q < W; ++q) {
        float gq;
        if (q == rank) gq = __ldcg(g + i);
        else if constexpr (sizeof(TT) == 4) gq = __ldcg(recv + q * P.slot_elems + rbase + i);
        else gq = __bfloat162float(recv[q * P.slot_elems + rbase + i]);
        gi = q == 0 ? gq : gi + gq;
      }
      if (clip > 0.f) gi = fminf(fmaxf(gi, -clip), clip);
      const float mi = m[i] + (1.f - beta1) * (gi - m[i]);
      const float vi = v[i] * beta2 + (1.f - beta2) * gi * gi;
      const float pn = p_loc[i] - ss * (mi / (sqrtf(vi) / bc + eps));
      m[i] = mi; v[i] = vi;
#pragma unroll
      for (int q = 0; q < W; ++q) P.param[q][i] = pn;
    }
  }
  // all my reads are done and my stores are on their way: one system fence per block (cumulative over the block's
  // accesses through the barrier), count blocks, last block runs the exit barrier and advances the epochs
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence_system();
    s_last = (atomicAdd(mypad + PAD_DONE_COUNTER, 1) == (int)gridDim.x - 1);
  }
  __syncthreads();
  if (s_last) {
    if (threadIdx.x == 0) __threadfence_system();
    __syncthreads();
    if (threadIdx.x < W) {
      st_release_sys(P.pad[threadIdx.x] + PAD_DONE + rank, e);
      while (ld_acquire_sys(mypad + PAD_DONE + threadIdx.x) < e) { }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      mypad[PAD_DONE_COUNTER] = 0; mypad[PAD_EPOCH] = e;
      for (int k = 1; k < P.n_wait; ++k) P.wait_pad[k][PAD_EPOCH] = P.wait_pad[k][PAD_EPOCH] + 1;
    }
  }
}

__global__ void mean_pixels_kernel(const float* __restrict__ feat, int64_t P, int64_t D, float* __restrict__ out) {
  int64_t b = blockIdx.y;
  int64_t d = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (d >= D) return;
  const float* src = feat + b * P * D + d;
  float s = 0.f;
  for (int64_t pz = 0; pz < P; ++pz) s += src[pz * D];
  out[b * D + d] = s / (float)P;
}

}  // namespace

extern "C" {

int32_t sn_gather_pack_fwd(const int64_t* captions, int64_t cap_ld, const float* table, int64_t E,
                           const float* features, int64_t feat_ld, int32_t has_feat,
                           const int32_t* row_b, const int32_t* row_t, const int32_t* tok_override,
                           int64_t N, float* X, int64_t ldx, float p_drop, uint64_t seed, const uint64_t* seed_dev,
                           void* Xb, int64_t ldxb, void* stream) {
  SN_REQUIRE(N >= 0 && E > 0 && (X || Xb), "sn_gather_pack_fwd: bad dims N=%lld E=%lld", (long long)N, (long long)E);
  SN_REQUIRE(!X || ldx >= E, "sn_gather_pack_fwd: ldx=%lld < E", (long long)ldx);
  SN_REQUIRE(!Xb || ldxb >= E, "sn_gather_pack_fwd: ldxb=%lld < E", (long long)ldxb);
  SN_REQUIRE(p_drop >= 0.f && p_drop < 1.f, "sn_gather_pack_fwd: dropout p=%f out of [0,1)", p_drop);
  SN_REQUIRE(!has_feat || features, "sn_gather_pack_fwd: has_feat without features");
  if (N == 0) return 0;
  float inv_keep = 1.f / (1.f - p_drop);
  unsigned grid = (unsigned)((N + 7) / 8);
  gather_pack_fwd_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(captions, cap_ld, table, (int)E, features, feat_ld,
                                                                 has_feat, row_b, row_t, tok_override, N, X, ldx,
                                                                 p_drop, inv_keep, seed, seed_dev,
                                                                 (__nv_bfloat16*)Xb, ldxb, Xb ? (int)ldxb : (int)E);
  return sn::check_launch("sn_gather_pack_fwd");
}

int32_t sn_gather_pack_bwd(const int64_t* captions, int64_t cap_ld, float* dtable, int64_t E,
                           float* dfeatures, int64_t feat_ld, int32_t has_feat, const int32_t* row_b,
                           const int32_t* row_t, const int32_t* tok_override, int64_t N,
                           const float* dX, int64_t ldx, float p_drop, uint64_t seed, const uint64_t* seed_dev,
                           int64_t V, int32_t* ws_int, float* ws_part, void* stream) {
  SN_REQUIRE(N >= 0 && E > 0 && ldx >= E && V > 0, "sn_gather_pack_bwd: bad dims");
  SN_REQUIRE(p_drop >= 0.f && p_drop < 1.f, "sn_gather_pack_bwd: dropout p=%f out of [0,1)", p_drop);
  SN_REQUIRE(N < (int64_t)1 << 30, "sn_gather_pack_bwd: N=%lld rows", (long long)N);
  if (N == 0) return 0;
  SN_REQUIRE(ws_int && ws_part, "sn_gather_pack_bwd: null work space");
  if (int32_t rc = sn_embed_plan(captions, cap_ld, has_feat, row_b, row_t, tok_override, N, V, ws_int, stream)) return rc;
  return sn_embed_grad(dtable, E, dfeatures, feat_ld, has_feat, row_b, row_t, tok_override, N, dX, ldx, p_drop, seed,
                       seed_dev, V, ws_int, ws_part, 0, stream);
}

namespace {
struct EmbedWs {      // layout of ws_int: see sn100.h
  int32_t *cnt, *start, *cursor, *cstart, *tok32, *perm, *sorted;
  EmbedWs(int32_t* ws, int64_t V, int64_t N)
      : cnt(ws), start(cnt + V), cursor(start + V + 1), cstart(cursor + V), tok32(cstart + V), perm(tok32 + N),
        sorted(perm + N) {}
};
}  // namespace

int32_t sn_embed_plan(const int64_t* captions, int64_t cap_ld, int32_t has_feat, const int32_t* row_b,
                      const int32_t* row_t, const int32_t* tok_override, int64_t N, int64_t V, int32_t* ws_int,
                      void* stream) {
  SN_REQUIRE(N >= 0 && N < (int64_t)1 << 30 && V > 0, "sn_embed_plan: bad dims N=%lld V=%lld", (long long)N, (long long)V);
  if (N == 0) return 0;
  SN_REQUIRE(ws_int, "sn_embed_plan: null work space");
  cudaStream_t st = (cudaStream_t)stream;
  EmbedWs w(ws_int, V, N);
  SN_CUDA(cudaMemsetAsync(w.cnt, 0, sizeof(int32_t) * (size_t)V, st));
  const unsigned g_rows = (unsigned)((N + 255) / 256);
  embed_count_kernel<<<g_rows, 256, 0, st>>>(captions, cap_ld, has_feat, row_b, row_t, tok_override, N, w.tok32, w.cnt);
  embed_scan_kernel<<<1, 1024, 0, st>>>(w.cnt, V, w.start, w.cursor, w.cstart);
  embed_place_kernel<<<g_rows, 256, 0, st>>>(w.tok32, N, w.cursor, w.perm);
  embed_order_kernel<<<g_rows, 256, 0, st>>>(w.tok32, w.start, w.perm, N, V, w.sorted);
  return sn::check_launch("sn_embed_plan");
}

int32_t sn_embed_grad(float* dtable, int64_t E, float* dfeatures, int64_t feat_ld, int32_t has_feat,
                      const int32_t* row_b, const int32_t* row_t, const int32_t* tok_override, int64_t N,
                      const float* dX, int64_t ldx, float p_drop, uint64_t seed, const uint64_t* seed_dev, int64_t V,
                      const int32_t* ws_int, float* ws_part, int32_t wide, void* stream) {
  SN_REQUIRE(N >= 0 && N < (int64_t)1 << 30 && E > 0 && ldx >= E && V > 0, "sn_embed_grad: bad dims");
  SN_REQUIRE(p_drop >= 0.f && p_drop < 1.f, "sn_embed_grad: dropout p=%f out of [0,1)", p_drop);
  if (N == 0) return 0;
  SN_REQUIRE(ws_int && ws_part, "sn_embed_grad: null work space");
  cudaStream_t st = (cudaStream_t)stream;
  float inv_keep = 1.f / (1.f - p_drop);
  if (has_feat && dfeatures)
    gather_pack_bwd_kernel<<<(unsigned)((N + 7) / 8), 256, 0, st>>>(nullptr, 0, dtable, (int)E, dfeatures,
                                                                     feat_ld, has_feat, row_b, row_t, tok_override, N,
                                                                     dX, ldx, p_drop, inv_keep, seed, seed_dev);
  EmbedWs w(const_cast<int32_t*>(ws_int), V, N);
  if (wide && E <= 512)
    embed_chunk_wide_kernel<<<(unsigned)N, (unsigned)((E + 31) / 32 * 32), 0, st>>>(
        w.tok32, w.start, w.cstart, w.sorted, V, tok_override, dX, ldx, (int)E, p_drop, inv_keep, seed, seed_dev,
        dtable, ws_part);
  else
    embed_chunk_kernel<<<(unsigned)((N + 7) / 8), 256, 0, st>>>(w.tok32, w.start, w.cstart, w.sorted, V, tok_override,
                                                                 dX, ldx, (int)E, p_drop, inv_keep, seed, seed_dev,
                                                                 dtable, ws_part);
  embed_combine_kernel<<<(unsigned)((V + 7) / 8), 256, 0, st>>>(w.cnt, w.cstart, V, (int)E, ws_part, dtable);
  return sn::check_launch("sn_embed_grad");
}

int32_t sn_softmax_nll(const float* logits, int64_t N, int64_t V, int64_t ld, const int64_t* targets,
                       float* row_loss, float* dlogits, int64_t ldd, float grad_scale, const float* row_weight,
                       int64_t* argmax, int32_t* top5hit, void* dlogits_bf16, int64_t lddb, void* stream) {
  SN_REQUIRE(N >= 0 && V > 0 && ld >= V, "sn_softmax_nll: bad dims");
  SN_REQUIRE(!dlogits_bf16 || lddb >= V, "sn_softmax_nll: lddb < V");
  if (N == 0) return 0;
  size_t smem = (size_t)V * sizeof(float);
  int use_smem = smem <= 200 * 1024;
  if (use_smem && smem > 48 * 1024) {
    static thread_local size_t configured = 0;
    if (configured < smem) {
      SN_CUDA(cudaFuncSetAttribute(softmax_nll_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
      configured = 200 * 1024;
    }
  }
  softmax_nll_kernel<<<(unsigned)N, 256, use_smem ? smem : 0, (cudaStream_t)stream>>>(
      logits, V, ld, targets, row_loss, dlogits, ldd, grad_scale, row_weight, argmax, top5hit, use_smem,
      (__nv_bfloat16*)dlogits_bf16, lddb);
  return sn::check_launch("sn_softmax_nll");
}

int32_t sn_reduce_sum(const float* x, int64_t N, float scale, const float* row_weight, float* out, int32_t accumulate,
                      void* stream) {
  SN_REQUIRE(N >= 0 && out, "sn_reduce_sum: bad args");
  reduce_sum_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(x, N, scale, row_weight, out, accumulate);
  return sn::check_launch("sn_reduce_sum");
}

int32_t sn_adam_clamp(float* p, float* g, float* m, float* v, int32_t n_ranges, const int64_t* ranges,
                      const float* step_size, const float* bc2_sqrt, float beta1, float beta2, float eps,
                      float clip, void* stream) {
  SN_REQUIRE(n_ranges >= 0, "sn_adam_clamp: n_ranges < 0");
  int done = 0;
  while (done < n_ranges) {
    AdamRanges R;
    R.n = 0;
    R.chunk_start[0] = 0;
    while (done < n_ranges && R.n < AdamRanges::MAX) {
      int64_t off = ranges[2 * done], len = ranges[2 * done + 1];
      SN_REQUIRE(off >= 0 && len >= 0 && len < ADAM_MAX_LEN, "sn_adam_clamp: bad range %d", done);
      R.off[R.n] = off; R.len[R.n] = (int32_t)len;
      R.step_size[R.n] = step_size[done]; R.bc2_sqrt[R.n] = bc2_sqrt[done];
      R.chunk_start[R.n + 1] = R.chunk_start[R.n] + (len + ADAM_CHUNK - 1) / ADAM_CHUNK;
      ++R.n; ++done;
    }
    int64_t chunks = R.chunk_start[R.n];
    if (chunks == 0) continue;
    int64_t cap = (int64_t)sn::dev_info().sm_count * 8;
    unsigned grid = (unsigned)(chunks < cap ? chunks : cap);
    adam_clamp_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(p, g, m, v, R, nullptr, beta1, beta2, eps, clip);
    int32_t rc = sn::check_launch("sn_adam_clamp");
    if (rc) return rc;
  }
  return 0;
}

int32_t sn_adam_clamp_dev(float* p, float* g, float* m, float* v, int32_t n_ranges, const int64_t* ranges,
                          const int32_t* step_idx, int32_t* steps_dev, const float* lr_dev, float* coef_ws,
                          float beta1, float beta2, float eps, float clip, void* stream) {
  return sn_adam_clamp_dev_ex(p, g, m, v, n_ranges, ranges, step_idx, steps_dev, lr_dev, coef_ws, beta1, beta2, eps,
                              clip, 0, stream);
}

int32_t sn_adam_clamp_dev_ex(float* p, float* g, float* m, float* v, int32_t n_ranges, const int64_t* ranges,
                             const int32_t* step_idx, int32_t* steps_dev, const float* lr_dev, float* coef_ws,
                             float beta1, float beta2, float eps, float clip, int32_t max_ctas, void* stream) {
  SN_REQUIRE(max_ctas >= 0, "sn_adam_clamp_dev: max_ctas < 0");
  SN_REQUIRE(n_ranges >= 0 && n_ranges <= AdamRanges::MAX, "sn_adam_clamp_dev: at most %d ranges per call", AdamRanges::MAX);
  SN_REQUIRE(steps_dev && lr_dev && coef_ws, "sn_adam_clamp_dev: null argument");
  if (n_ranges == 0) return 0;
  AdamRanges R;
  R.n = n_ranges;
  R.chunk_start[0] = 0;
  for (int i = 0; i < n_ranges; ++i) {
    SN_REQUIRE(ranges[2 * i] >= 0 && ranges[2 * i + 1] >= 0 && ranges[2 * i + 1] < ADAM_MAX_LEN, "sn_adam_clamp_dev: bad range %d", i);
    R.off[i] = ranges[2 * i]; R.len[i] = (int32_t)ranges[2 * i + 1]; R.step_idx[i] = step_idx[i];
    R.step_size[i] = 0.f; R.bc2_sqrt[i] = 1.f;
    R.chunk_start[i + 1] = R.chunk_start[i] + (R.len[i] + ADAM_CHUNK - 1) / ADAM_CHUNK;
  }
  cudaStream_t st = (cudaStream_t)stream;
  adam_prepare_kernel<<<1, AdamRanges::MAX, 0, st>>>(R, steps_dev, lr_dev, coef_ws, beta1, beta2);
  int64_t chunks = R.chunk_start[R.n];
  if (chunks == 0) return sn::check_launch("sn_adam_clamp_dev");
  int64_t cap = (int64_t)sn::dev_info().sm_count * 8;
  if (max_ctas > 0 && max_ctas < cap) cap = max_ctas;
  unsigned grid = (unsigned)(chunks < cap ? chunks : cap);
  adam_clamp_kernel<<<grid, 256, 0, st>>>(p, g, m, v, R, coef_ws, beta1, beta2, eps, clip);
  return sn::check_launch("sn_adam_clamp_dev");
}

int32_t sn_enable_peer_access(int32_t peer_device) {
  int cur = 0;
  SN_CUDA(cudaGetDevice(&cur));
  if (peer_device == cur) return 0;
  int can = 0;
  SN_CUDA(cudaDeviceCanAccessPeer(&can, cur, peer_device));
  SN_REQUIRE(can, "sn_enable_peer_access: device %d cannot access peer %d", cur, peer_device);
  cudaError_t e = cudaDeviceEnablePeerAccess(peer_device, 0);
  if (e == cudaErrorPeerAccessAlreadyEnabled) { cudaGetLastError(); return 0; }
  if (e != cudaSuccess) return sn::fail((int32_t)e, "cudaDeviceEnablePeerAccess(%d): %s", peer_device, cudaGetErrorString(e));
  return 0;
}

int32_t sn_dp_adam_fused(int32_t world, int32_t rank, void* const* grad_ptrs, void* const* param_ptrs,
                         void* const* pad_ptrs, float* m, float* v, int32_t n_ranges, const int64_t* ranges,
                         const int32_t* step_idx, int32_t* steps_dev, const float* lr_dev, float* coef_ws, float beta1,
                         float beta2, float eps, float clip, void* stream) {
  SN_REQUIRE(world >= 1 && world <= 8 && rank >= 0 && rank < world, "sn_dp_adam_fused: bad world/rank %d/%d", world, rank);
  SN_REQUIRE(n_ranges >= 0 && n_ranges <= AdamRanges::MAX, "sn_dp_adam_fused: at most %d ranges per call", AdamRanges::MAX);
  SN_REQUIRE(grad_ptrs && param_ptrs && pad_ptrs && steps_dev && lr_dev && coef_ws && m && v, "sn_dp_adam_fused: null argument");
  DpPeers P;
  memset(&P, 0, sizeof(P));
  P.world = world; P.rank = rank;
  for (int q = 0; q < 8; ++q) {
    P.grad[q] = q < world ? (float*)grad_ptrs[q] : nullptr;
    P.param[q] = q < world ? (float*)param_ptrs[q] : nullptr;
    P.pad[q] = q < world ? (int*)pad_ptrs[q] : nullptr;
    SN_REQUIRE(q >= world || (P.grad[q] && P.param[q] && P.pad[q]), "sn_dp_adam_fused: null peer pointer %d", q);
  }
  AdamRanges R;
  R.n = n_ranges;
  R.chunk_start[0] = 0;
  for (int i = 0; i < n_ranges; ++i) {
    SN_REQUIRE(ranges[2 * i] >= 0 && ranges[2 * i + 1] >= 0 && ranges[2 * i + 1] < ADAM_MAX_LEN, "sn_dp_adam_fused: bad range %d", i);
    R.off[i] = ranges[2 * i]; R.len[i] = (int32_t)ranges[2 * i + 1]; R.step_idx[i] = step_idx[i];
    R.step_size[i] = 0.f; R.bc2_sqrt[i] = 1.f;
    // chunks on the absolute ADAM_CHUNK grid of the arena (ownership must not depend on the active set, see the kernel)
    R.chunk_start[i + 1] = R.chunk_start[i] +
        (R.len[i] > 0 ? (R.off[i] + R.len[i] - 1) / ADAM_CHUNK - R.off[i] / ADAM_CHUNK + 1 : 0);
  }
  cudaStream_t st = (cudaStream_t)stream;
  if (n_ranges > 0) adam_prepare_kernel<<<1, AdamRanges::MAX, 0, st>>>(R, steps_dev, lr_dev, coef_ws, beta1, beta2);
  // every rank launches the same grid even when it owns no chunk: the kernel is also the cross-GPU barrier
  int64_t mine = (R.chunk_start[R.n] + world - 1) / world;
  // persistent: at most 3 CTAs per SM loop over the slots (every CTA ends with a system-scope fence and an atomic)
  int64_t cap = (int64_t)sn::dev_info().sm_count * 3;
  unsigned grid = (unsigned)(mine < 1 ? 1 : (mine < cap ? mine : cap));
  static const int dbg = [] { const char* e = getenv("SN_DP_DEBUG"); return e ? atoi(e) : 0; }();
#define SN_DP_LAUNCH(WW) dp_adam_fused_kernel<WW><<<grid, 256, 0, st>>>(P, R, coef_ws, m, v, beta1, beta2, eps, clip, dbg)
  switch (world) {
    case 1: SN_DP_LAUNCH(1); break;
    case 2: SN_DP_LAUNCH(2); break;
    case 3: SN_DP_LAUNCH(3); break;
    case 4: SN_DP_LAUNCH(4); break;
    case 5: SN_DP_LAUNCH(5); break;
    case 6: SN_DP_LAUNCH(6); break;
    case 7: SN_DP_LAUNCH(7); break;
    default: SN_DP_LAUNCH(8); break;
  }
#undef SN_DP_LAUNCH
  return sn::check_launch("sn_dp_adam_fused");
}

static int32_t dp_fill_ranges(AdamRanges& R, int32_t n_ranges, const int64_t* ranges, const int32_t* step_idx, const char* who) {
  SN_REQUIRE(n_ranges >= 0 && n_ranges <= AdamRanges::MAX, "%s: at most %d ranges per call", who, AdamRanges::MAX);
  R.n = n_ranges;
  R.chunk_start[0] = 0;
  for (int i = 0; i < n_ranges; ++i) {
    SN_REQUIRE(ranges[2 * i] >= 0 && ranges[2 * i + 1] >= 0 && ranges[2 * i + 1] < ADAM_MAX_LEN, "%s: bad range %d", who, i);
    R.off[i] = ranges[2 * i]; R.len[i] = (int32_t)ranges[2 * i + 1]; R.step_idx[i] = step_idx ? step_idx[i] : 0;
    R.step_size[i] = 0.f; R.bc2_sqrt[i] = 1.f;
    R.chunk_start[i + 1] = R.chunk_start[i] +
        (R.len[i] > 0 ? (R.off[i] + R.len[i] - 1) / ADAM_CHUNK - R.off[i] / ADAM_CHUNK + 1 : 0);
  }
  return 0;
}

int64_t sn_dp_slot_elems(int64_t arena_elems, int32_t world) {
  if (arena_elems < 0 || world < 1) return -1;
  int64_t chunks = (arena_elems + ADAM_CHUNK - 1) / ADAM_CHUNK;
  return ((chunks + world - 1) / world) * ADAM_CHUNK;
}

int32_t sn_dp_push(int32_t world, int32_t rank, const float* grad, void* const* recv_ptrs, int64_t slot_elems,
                   int32_t elem_size, void* const* pad_ptrs, int32_t n_ranges, const int64_t* ranges, int32_t max_ctas,
                   void* stream) {
  SN_REQUIRE(world >= 1 && world <= 8 && rank >= 0 && rank < world, "sn_dp_push: bad world/rank %d/%d", world, rank);
  SN_REQUIRE(grad && recv_ptrs && pad_ptrs && ranges, "sn_dp_push: null argument");
  SN_REQUIRE(elem_size == 4 || elem_size == 2, "sn_dp_push: elem_size must be 4 (fp32) or 2 (bf16)");
  SN_REQUIRE(slot_elems > 0 && slot_elems % ADAM_CHUNK == 0, "sn_dp_push: slot_elems must be a positive multiple of %d", ADAM_CHUNK);
  DpPeers P;
  memset(&P, 0, sizeof(P));
  P.world = world; P.rank = rank; P.slot_elems = slot_elems;
  for (int q = 0; q < world; ++q) {
    P.recv[q] = recv_ptrs[q]; P.pad[q] = (int*)pad_ptrs[q];
    SN_REQUIRE(P.recv[q] && P.pad[q], "sn_dp_push: null peer pointer %d", q);
  }
  AdamRanges R;
  if (int32_t rc = dp_fill_ranges(R, n_ranges, ranges, nullptr, "sn_dp_push")) return rc;
  for (int i = 0; i < n_ranges; ++i)
    SN_REQUIRE(R.len[i] == 0 || (R.off[i] + R.len[i] - 1) / ADAM_CHUNK / world < slot_elems / ADAM_CHUNK,
               "sn_dp_push: range %d does not fit the receive slots", i);
  // every rank launches (the kernel also raises the ARRIVE flags); a light grid: the NVLink stores, not the SMs, set
  // the pace, and the producing stream's neighbours (weight-gradient GEMMs) keep their SMs
  int64_t chunks = R.chunk_start[R.n];
  int64_t cap = (int64_t)sn::dev_info().sm_count;
  if (max_ctas > 0 && max_ctas < cap) cap = max_ctas;      // background exchange under the backward: leave the GEMMs their SMs
  int64_t want = (chunks + DP_SUB - 1) / DP_SUB;
  unsigned grid = (unsigned)(want < 1 ? 1 : (want < cap ? want : cap));
  cudaStream_t st = (cudaStream_t)stream;
  if (elem_size == 4) dp_push_kernel<float><<<grid, 256 * DP_SUB, 0, st>>>(P, R, grad);
  else dp_push_kernel<__nv_bfloat16><<<grid, 256 * DP_SUB, 0, st>>>(P, R, grad);
  return sn::check_launch("sn_dp_push");
}

int32_t sn_dp_adam_recv(int32_t world, int32_t rank, float* grad, void* const* param_ptrs, void* recv, int64_t slot_elems,
                        int32_t elem_size, void* const* pad_ptrs, void* const* wait_pads, int32_t n_wait, float* m, float* v,
                        int32_t n_ranges, const int64_t* ranges, const int32_t* step_idx, int32_t* steps_dev,
                        const float* lr_dev, float* coef_ws, float beta1, float beta2, float eps, float clip,
                        int32_t max_ctas, void* stream) {
  SN_REQUIRE(world >= 1 && world <= 8 && rank >= 0 && rank < world, "sn_dp_adam_recv: bad world/rank %d/%d", world, rank);
  SN_REQUIRE(grad && param_ptrs && recv && pad_ptrs && wait_pads && steps_dev && lr_dev && coef_ws && m && v && ranges && step_idx,
             "sn_dp_adam_recv: null argument");
  SN_REQUIRE(elem_size == 4 || elem_size == 2, "sn_dp_adam_recv: elem_size must be 4 (fp32) or 2 (bf16)");
  SN_REQUIRE(n_wait >= 1 && n_wait <= 4, "sn_dp_adam_recv: 1..4 push buckets per call (got %d)", n_wait);
  SN_REQUIRE(slot_elems > 0 && slot_elems % ADAM_CHUNK == 0, "sn_dp_adam_recv: slot_elems must be a positive multiple of %d", ADAM_CHUNK);
  SN_REQUIRE(n_ranges >= 1, "sn_dp_adam_recv: no ranges");
  DpPeers P;
  memset(&P, 0, sizeof(P));
  P.world = world; P.rank = rank; P.slot_elems = slot_elems; P.n_wait = n_wait;
  for (int q = 0; q < world; ++q) {
    P.param[q] = (float*)param_ptrs[q]; P.pad[q] = (int*)pad_ptrs[q];
    SN_REQUIRE(P.param[q] && P.pad[q], "sn_dp_adam_recv: null peer pointer %d", q);
  }
  P.grad[rank] = grad;
  P.recv[rank] = recv;
  for (int k = 0; k < n_wait; ++k) {
    P.wait_pad[k] = (int*)wait_pads[k];
    SN_REQUIRE(P.wait_pad[k], "sn_dp_adam_recv: null wait pad %d", k);
  }
  SN_REQUIRE(P.wait_pad[0] == P.pad[rank], "sn_dp_adam_recv: pad_ptrs must be every rank's pad of wait bucket 0");
  AdamRanges R;
  if (int32_t rc = dp_fill_ranges(R, n_ranges, ranges, step_idx, "sn_dp_adam_recv")) return rc;
  // chunk_start = prefix of the chunks THIS rank owns in each range (absolute chunk id % world == rank)
  for (int i = 0; i < n_ranges; ++i) {
    int64_t own = 0;
    if (R.len[i] > 0) {
      const int64_t a0 = R.off[i] / ADAM_CHUNK, a1 = (R.off[i] + R.len[i] - 1) / ADAM_CHUNK;
      const int64_t first = a0 + ((rank - a0) % world + world) % world;
      own = first <= a1 ? (a1 - first) / world + 1 : 0;
      SN_REQUIRE(a1 / world < slot_elems / ADAM_CHUNK, "sn_dp_adam_recv: range %d does not fit the receive slots", i);
    }
    R.chunk_start[i + 1] = R.chunk_start[i] + own;
  }
  cudaStream_t st = (cudaStream_t)stream;
  adam_prepare_kernel<<<1, AdamRanges::MAX, 0, st>>>(R, steps_dev, lr_dev, coef_ws, beta1, beta2);
  // every rank launches (the kernel is also the exit barrier), also one that owns no chunk of these ranges
  int64_t mine = (R.chunk_start[R.n] + DP_RSUB - 1) / DP_RSUB;
  int64_t cap = (int64_t)sn::dev_info().sm_count * 2;
  if (max_ctas > 0 && max_ctas < cap) cap = max_ctas;
  unsigned grid = (unsigned)(mine < 1 ? 1 : (mine < cap ? mine : cap));
  const float* p_loc = P.param[rank];
#define SN_DP_LAUNCH(WW)                                                                                                   \
  if (elem_size == 4) dp_recv_adam_kernel<WW, float><<<grid, 256 * DP_RSUB, 0, st>>>(P, R, coef_ws, grad, (const float*)recv, p_loc, m, v, beta1, beta2, eps, clip); \
  else dp_recv_adam_kernel<WW, __nv_bfloat16><<<grid, 256 * DP_RSUB, 0, st>>>(P, R, coef_ws, grad, (const __nv_bfloat16*)recv, p_loc, m, v, beta1, beta2, eps, clip)
  switch (world) {
    case 1: SN_DP_LAUNCH(1); break;
    case 2: SN_DP_LAUNCH(2); break;
    case 3: SN_DP_LAUNCH(3); break;
    case 4: SN_DP_LAUNCH(4); break;
    case 5: SN_DP_LAUNCH(5); break;
    case 6: SN_DP_LAUNCH(6); break;
    case 7: SN_DP_LAUNCH(7); break;
    default: SN_DP_LAUNCH(8); break;
  }
#undef SN_DP_LAUNCH
  return sn::check_launch("sn_dp_adam_recv");
}

int32_t sn_mean_pixels(const float* feat, int64_t B, int64_t P, int64_t D, float* out, void* stream) {
  SN_REQUIRE(B >= 0 && P > 0 && D > 0, "sn_mean_pixels: bad dims");
  if (B == 0) return 0;
  dim3 grid((unsigned)((D + 255) / 256), (unsigned)B);
  mean_pixels_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(feat, P, D, out);
  return sn::check_launch("sn_mean_pixels");
}

}  // extern "C"
