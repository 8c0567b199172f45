// fp32 FFMA GEMM (SN_PREC_F32): the exact-fp32 arithmetic path and the validation reference for the
// tcgen05 GEMMs.  128x128x8 tiles, 256 threads, 8x8 register micro-tiles, generic operand strides so
// that NT / NN / TN all run without materialised transposes.
#include <cooperative_groups.h>
#include <cuda_bf16.h>

#include "sn_common.cuh"

namespace cg = cooperative_groups;

namespace {

struct GemmArgs {
  int64_t M, N, K;
  const float* A; int64_t sam, sak;   // A(m,k) = A[m*sam + k*sak]
  const float* B; int64_t sbk, sbn;   // B(k,n) = B[k*sbk + n*sbn]
  float* C; int64_t ldc;
  const float* bias; float beta;
  int64_t strideA, strideB, strideC, strideBias;
};

constexpr int BM = 128, BN = 128, BK = 8;

// one thread's share (4 elements) of a [major x BK] operand tile: fetched into registers first so that the
// global loads of tile i+1 are in flight while tile i is being multiplied (software pipelining)
struct Frag { float v[4]; };

__device__ __forceinline__ Frag fetch_tile(const float* __restrict__ P, int64_t s_major, int64_t s_k, int64_t major0,
                                           int64_t k0, int64_t major_lim, int64_t k_lim, int tid) {
  Frag f;
  f.v[0] = f.v[1] = f.v[2] = f.v[3] = 0.f;
  if (s_k == 1) {
    // k contiguous: thread -> (major = tid/2, 4 consecutive k)
    int mj = tid >> 1, kk = (tid & 1) * 4;
    int64_t gm = major0 + mj, gk = k0 + kk;
    if (gm < major_lim) {
      const float* src = P + gm * s_major + gk;
      if (gk + 3 < k_lim && ((reinterpret_cast<uintptr_t>(src) & 15) == 0)) {
        float4 t = __ldg(reinterpret_cast<const float4*>(src));
        f.v[0] = t.x; f.v[1] = t.y; f.v[2] = t.z; f.v[3] = t.w;
      } else {
#pragma unroll
        for (int j = 0; j < 4; ++j) if (gk + j < k_lim) f.v[j] = __ldg(src + j);
      }
    }
  } else {
    // major contiguous (s_major == 1): thread -> (k = tid/32, 4 consecutive major)
    int kk = tid >> 5, mj = (tid & 31) * 4;
    int64_t gm = major0 + mj, gk = k0 + kk;
    if (gk < k_lim) {
      const float* src = P + gk * s_k + gm * s_major;
      if (s_major == 1 && gm + 3 < major_lim && ((reinterpret_cast<uintptr_t>(src) & 15) == 0)) {
        float4 t = __ldg(reinterpret_cast<const float4*>(src));
        f.v[0] = t.x; f.v[1] = t.y; f.v[2] = t.z; f.v[3] = t.w;
      } else {
#pragma unroll
        for (int j = 0; j < 4; ++j) if (gm + j < major_lim) f.v[j] = __ldg(src + j * s_major);
      }
    }
  }
  return f;
}

__device__ __forceinline__ void store_tile(float (*S)[BM + 4], const Frag& f, int64_t s_k, int tid) {
  if (s_k == 1) {
    int mj = tid >> 1, kk = (tid & 1) * 4;
#pragma unroll
    for (int j = 0; j < 4; ++j) S[kk + j][mj] = f.v[j];
  } else {
    int kk = tid >> 5, mj = (tid & 31) * 4;
    *reinterpret_cast<float4*>(&S[kk][mj]) = make_float4(f.v[0], f.v[1], f.v[2], f.v[3]);
  }
}

__global__ void __launch_bounds__(256) gemm_simt_kernel(GemmArgs g) {
  __shared__ __align__(16) float As[BK][BM + 4];
  __shared__ __align__(16) float Bs[BK][BN + 4];
  const int tid = threadIdx.x;
  const int64_t m0 = (int64_t)blockIdx.y * BM, n0 = (int64_t)blockIdx.x * BN;
  const float* A = g.A + blockIdx.z * g.strideA;
  const float* B = g.B + blockIdx.z * g.strideB;
  float* C = g.C + blockIdx.z * g.strideC;
  const float* bias = g.bias ? g.bias + blockIdx.z * g.strideBias : nullptr;

  const int ty = tid >> 4, tx = tid & 15;
  float acc[8][8];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;

  Frag fa = fetch_tile(A, g.sam, g.sak, m0, 0, g.M, g.K, tid);
  Frag fb = fetch_tile(B, g.sbn, g.sbk, n0, 0, g.N, g.K, tid);
  for (int64_t k0 = 0; k0 < g.K; k0 += BK) {
    store_tile(As, fa, g.sak, tid);
    store_tile(Bs, fb, g.sbk, tid);
    __syncthreads();
    if (k0 + BK < g.K) {      // next tile's global loads fly while this tile is multiplied
      fa = fetch_tile(A, g.sam, g.sak, m0, k0 + BK, g.M, g.K, tid);
      fb = fetch_tile(B, g.sbn, g.sbk, n0, k0 + BK, g.N, g.K, tid);
    }
#pragma unroll
    for (int k = 0; k < BK; ++k) {
      float4 a0 = *reinterpret_cast<const float4*>(&As[k][ty * 4]);
      float4 a1 = *reinterpret_cast<const float4*>(&As[k][64 + ty * 4]);
      float4 b0 = *reinterpret_cast<const float4*>(&Bs[k][tx * 4]);
      float4 b1 = *reinterpret_cast<const float4*>(&Bs[k][64 + tx * 4]);
      float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
      float b[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }

#pragma unroll
  for (int i = 0; i < 8; ++i) {
    int64_t m = m0 + (i < 4 ? ty * 4 + i : 64 + ty * 4 + (i - 4));
    if (m >= g.M) continue;
#pragma unroll
    for (int jh = 0; jh < 2; ++jh) {
      int64_t n = n0 + jh * 64 + tx * 4;
      float* dst = C + m * g.ldc + n;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        if (n + j < g.N) {
          float v = acc[i][jh * 4 + j];
          if (bias) v += bias[n + j];
          if (g.beta != 0.f) v += g.beta * dst[j];
          dst[j] = v;
        }
      }
    }
  }
}

// Skinny NT GEMM for decode steps (M <= 16 rows: live beams / a single image): weight-bandwidth bound, so one
// warp streams one weight row (coalesced, 128-bit) and dots it with all M input rows held in shared memory.
constexpr int SK_MAXM = 16;

__global__ void __launch_bounds__(256) gemm_skinny_nt_kernel(GemmArgs g) {
  extern __shared__ __align__(16) float xs[];      // [M][Kp]
  const int m0 = blockIdx.z * SK_MAXM;             // rows are processed 16 at a time (grid.z chunks)
  const int M = min(SK_MAXM, (int)g.M - m0), K = (int)g.K;
  const int Kp = (K + 3) & ~3;
  const float* A = g.A + blockIdx.y * g.strideA + (int64_t)m0 * g.sam;
  const float* B = g.B + blockIdx.y * g.strideB;
  float* C = g.C + blockIdx.y * g.strideC + (int64_t)m0 * g.ldc;
  const float* bias = g.bias ? g.bias + blockIdx.y * g.strideBias : nullptr;
  for (int i = threadIdx.x; i < M * Kp; i += 256) {
    int m = i / Kp, k = i - m * Kp;
    xs[i] = k < K ? A[(int64_t)m * g.sam + k] : 0.f;
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t n = (int64_t)blockIdx.x * 8 + warp;
  if (n >= g.N) return;
  const float* w = B + n * g.sbn;                  // row n of B[N,K] (k contiguous)
  float acc[SK_MAXM];
#pragma unroll
  for (int m = 0; m < SK_MAXM; ++m) acc[m] = 0.f;
  const bool vec = ((reinterpret_cast<uintptr_t>(w) & 15) == 0);
  if (vec) {
    for (int k = lane * 4; k < K; k += 128) {
      float4 wv;
      if (k + 3 < K) wv = __ldg(reinterpret_cast<const float4*>(w + k));
      else { wv.x = w[k]; wv.y = k + 1 < K ? w[k + 1] : 0.f; wv.z = k + 2 < K ? w[k + 2] : 0.f; wv.w = 0.f; }
#pragma unroll
      for (int m = 0; m < SK_MAXM; ++m) {
        if (m < M) {
          const float4 xv = *reinterpret_cast<const float4*>(xs + m * Kp + k);
          acc[m] = fmaf(wv.x, xv.x, fmaf(wv.y, xv.y, fmaf(wv.z, xv.z, fmaf(wv.w, xv.w, acc[m]))));
        }
      }
    }
  } else {
    for (int k = lane; k < K; k += 32) {
      const float wv = __ldg(w + k);
#pragma unroll
      for (int m = 0; m < SK_MAXM; ++m) if (m < M) acc[m] = fmaf(wv, xs[m * Kp + k], acc[m]);
    }
  }
#pragma unroll
  for (int m = 0; m < SK_MAXM; ++m) {
    if (m < M) {
      float v = sn::warp_sum(acc[m]);
      if (lane == 0) C[(int64_t)m * g.ldc + n] = v + (bias ? bias[n] : 0.f);
    }
  }
}

constexpr int CS_CLUSTER = 8;  // CTAs per column strip, one cluster: each sums 1/8 of the rows
constexpr int CS_LANES = 32;   // row lanes per CTA

__device__ __forceinline__ float to_f(float v) { return v; }
__device__ __forceinline__ float to_f(__nv_bfloat16 v) { return __bfloat162float(v); }

// grid (ceil(N/32), CS_CLUSTER); block 32 columns x CS_LANES row lanes.  The partial sums of the cluster's CTAs are
// added by rank 0 through distributed shared memory in rank order: every summation order is fixed, so the result is
// the same from run to run (bias gradients feed Adam, which turns last-bit differences into +-lr steps).
template <typename TIn>
__global__ void __cluster_dims__(1, CS_CLUSTER, 1) __launch_bounds__(32 * CS_LANES) colsum_kernel(const TIn* __restrict__ X, int64_t M, int64_t N,
                                                                 int64_t ldx, float* __restrict__ out, float beta) {
  __shared__ float part[CS_LANES][33];
  __shared__ float tot[32];
  cg::cluster_group cluster = cg::this_cluster();
  const int col = blockIdx.x * 32 + threadIdx.x;
  const int64_t chunk = (M + CS_CLUSTER - 1) / CS_CLUSTER;
  const int64_t r0 = (int64_t)blockIdx.y * chunk;
  const int64_t r1 = r0 + chunk < M ? r0 + chunk : M;
  float s = 0.f;
  if (col < N)
    for (int64_t m = r0 + threadIdx.y; m < r1; m += CS_LANES) s += to_f(X[m * ldx + col]);
  part[threadIdx.y][threadIdx.x] = s;
  __syncthreads();
  if (threadIdx.y == 0) {
    float t = 0.f;
#pragma unroll
    for (int j = 0; j < CS_LANES; ++j) t += part[j][threadIdx.x];
    tot[threadIdx.x] = t;
  }
  cluster.sync();
  if (cluster.block_rank() == 0 && threadIdx.y == 0 && col < N) {
    float t = 0.f;
#pragma unroll
    for (int r = 0; r < CS_CLUSTER; ++r) t += cluster.map_shared_rank(tot, r)[threadIdx.x];
    out[col] = beta == 0.f ? t : beta * out[col] + t;
  }
  cluster.sync();   // the other CTAs' shared memory stays alive until rank 0 has read it
}

// The same sums as colsum_kernel, bit for bit, with 16-byte loads: thread x reads VEC adjacent columns (8 bf16 or 4
// fp32), so a CTA covers 32 * VEC columns.  The order is unchanged: rows in CS_CLUSTER chunks, lane y summing rows
// r0+y, r0+y+32, ... in order, lanes added 0..31, ranks 0..CS_CLUSTER-1.  A strip's last columns past N are read one
// by one.  Needs X and ldx aligned to 16 bytes.
template <typename TIn>
__global__ void __cluster_dims__(1, CS_CLUSTER, 1) __launch_bounds__(32 * CS_LANES)
colsum_wide_kernel(const TIn* __restrict__ X, int64_t M, int64_t N, int64_t ldx, float* __restrict__ out, float beta) {
  constexpr int VEC = 16 / sizeof(TIn);
  constexpr int W = 32 * VEC;       // columns per CTA
  __shared__ float part[CS_LANES][W + 1];
  __shared__ float tot[W];
  cg::cluster_group cluster = cg::this_cluster();
  const int64_t c0 = (int64_t)blockIdx.x * W + threadIdx.x * VEC;
  const int64_t chunk = (M + CS_CLUSTER - 1) / CS_CLUSTER;
  const int64_t r0 = (int64_t)blockIdx.y * chunk;
  const int64_t r1 = r0 + chunk < M ? r0 + chunk : M;
  float s[VEC];
#pragma unroll
  for (int e = 0; e < VEC; ++e) s[e] = 0.f;
  if (c0 + VEC <= N) {
    for (int64_t m = r0 + threadIdx.y; m < r1; m += CS_LANES) {
      const uint4 raw = *reinterpret_cast<const uint4*>(X + m * ldx + c0);
      const TIn* x = reinterpret_cast<const TIn*>(&raw);
#pragma unroll
      for (int e = 0; e < VEC; ++e) s[e] += to_f(x[e]);
    }
  } else if (c0 < N) {
    for (int64_t m = r0 + threadIdx.y; m < r1; m += CS_LANES)
#pragma unroll
      for (int e = 0; e < VEC; ++e)
        if (c0 + e < N) s[e] += to_f(X[m * ldx + c0 + e]);
  }
#pragma unroll
  for (int e = 0; e < VEC; ++e) part[threadIdx.y][threadIdx.x * VEC + e] = s[e];
  __syncthreads();
  const int tid = threadIdx.y * 32 + threadIdx.x;
  if (tid < W) {
    float t = 0.f;
#pragma unroll
    for (int j = 0; j < CS_LANES; ++j) t += part[j][tid];
    tot[tid] = t;
  }
  cluster.sync();
  const int64_t col = (int64_t)blockIdx.x * W + tid;
  if (cluster.block_rank() == 0 && tid < W && col < N) {
    float t = 0.f;
#pragma unroll
    for (int r = 0; r < CS_CLUSTER; ++r) t += cluster.map_shared_rank(tot, r)[tid];
    out[col] = beta == 0.f ? t : beta * out[col] + t;
  }
  cluster.sync();   // the other CTAs' shared memory stays alive until rank 0 has read it
}

}  // namespace

extern "C" int32_t sn_gemm(int32_t op, int64_t M, int64_t N, int64_t K, const float* A, int64_t lda,
                           const float* B, int64_t ldb, float* C, int64_t ldc, const float* bias,
                           float beta, int32_t batch, int64_t strideA, int64_t strideB,
                           int64_t strideC, int64_t strideBias, void* stream) {
  SN_REQUIRE(op >= 0 && op <= 2, "sn_gemm: bad op %d", op);
  SN_REQUIRE(M >= 0 && N >= 0 && K >= 0 && batch >= 1, "sn_gemm: bad dims M=%lld N=%lld K=%lld batch=%d",
             (long long)M, (long long)N, (long long)K, batch);
  if (M == 0 || N == 0) return 0;
  SN_REQUIRE(A && B && C, "sn_gemm: null operand");
  GemmArgs g;
  g.M = M; g.N = N; g.K = K;
  g.A = A; g.B = B; g.C = C; g.ldc = ldc; g.bias = bias; g.beta = beta;
  g.strideA = strideA; g.strideB = strideB; g.strideC = strideC; g.strideBias = strideBias;
  if (op == SN_OP_NT) { g.sam = lda; g.sak = 1; g.sbk = 1; g.sbn = ldb; }
  else if (op == SN_OP_NN) { g.sam = lda; g.sak = 1; g.sbk = ldb; g.sbn = 1; }
  else { g.sam = 1; g.sak = lda; g.sbk = ldb; g.sbn = 1; }
  if (op == SN_OP_NT && M <= 8 * SK_MAXM && beta == 0.f) {
    // few rows (decode steps, per-time-step Linears): weight-bandwidth bound -> skinny kernel, 16 rows per CTA.z
    size_t smem = (size_t)(M < SK_MAXM ? M : SK_MAXM) * ((K + 3) & ~(int64_t)3) * sizeof(float);
    if (smem <= 96 * 1024) {
      if (smem > 48 * 1024) {
        static thread_local bool configured = false;
        if (!configured) {
          SN_CUDA(cudaFuncSetAttribute(gemm_skinny_nt_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024));
          configured = true;
        }
      }
      dim3 sgrid((unsigned)((N + 7) / 8), (unsigned)batch, (unsigned)((M + SK_MAXM - 1) / SK_MAXM));
      gemm_skinny_nt_kernel<<<sgrid, 256, smem, (cudaStream_t)stream>>>(g);
      return sn::check_launch("sn_gemm(skinny)");
    }
  }
  dim3 grid((unsigned)((N + BN - 1) / BN), (unsigned)((M + BM - 1) / BM), (unsigned)batch);
  gemm_simt_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(g);
  return sn::check_launch("sn_gemm");
}

namespace {
template <typename TIn>
int32_t colsum_launch(const TIn* X, int64_t M, int64_t N, int64_t ldx, float* out, float beta, int32_t wide,
                      void* stream) {
  SN_REQUIRE(M >= 0 && N >= 0, "sn_colsum: bad dims");
  if (N == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  if (M == 0 && beta == 0.f) {
    SN_CUDA(cudaMemsetAsync(out, 0, sizeof(float) * (size_t)N, st));
    return 0;
  }
  constexpr int VEC = 16 / sizeof(TIn);
  dim3 block(32, CS_LANES);
  if (wide && ((uintptr_t)X & 15) == 0 && ldx % VEC == 0) {
    dim3 grid((unsigned)((N + 32 * VEC - 1) / (32 * VEC)), CS_CLUSTER);
    colsum_wide_kernel<TIn><<<grid, block, 0, st>>>(X, M, N, ldx, out, beta);
  } else {
    dim3 grid((unsigned)((N + 31) / 32), CS_CLUSTER);
    colsum_kernel<TIn><<<grid, block, 0, st>>>(X, M, N, ldx, out, beta);
  }
  return sn::check_launch("sn_colsum");
}
}  // namespace

extern "C" int32_t sn_colsum(const float* X, int64_t M, int64_t N, int64_t ldx, float* out, float beta,
                             void* stream) {
  return colsum_launch<float>(X, M, N, ldx, out, beta, 0, stream);
}

extern "C" int32_t sn_colsum_bf16(const void* X, int64_t M, int64_t N, int64_t ldx, float* out, float beta,
                                  void* stream) {
  return colsum_launch<__nv_bfloat16>((const __nv_bfloat16*)X, M, N, ldx, out, beta, 0, stream);
}

extern "C" int32_t sn_colsum_ex(const float* X, int64_t M, int64_t N, int64_t ldx, float* out, float beta,
                                int32_t wide, void* stream) {
  return colsum_launch<float>(X, M, N, ldx, out, beta, wide, stream);
}

extern "C" int32_t sn_colsum_bf16_ex(const void* X, int64_t M, int64_t N, int64_t ldx, float* out, float beta,
                                     int32_t wide, void* stream) {
  return colsum_launch<__nv_bfloat16>((const __nv_bfloat16*)X, M, N, ldx, out, beta, wide, stream);
}
