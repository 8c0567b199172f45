// Decode-step kernels for FEW rows (single-image beam search: rows = live beams <= 8, forward_step on a handful of
// rows): at these sizes a decode step is a handful of matrix-VECTOR products, bound by one pass over the weights
// (35 MB fp32 at configs[1]) -- not GEMMs.  Each output feature is one warp-level dot product per row with the weight
// row streamed once with 128-bit loads; the R input rows (a few KB) are read through L1.
//   sn_skinny_linear : out[r, n] = bias[n] + W[n, :] . X[r, xoff(n) : xoff(n) + K]      (V / S stages, vocabulary C)
//   sn_decode_cell   : forward_step's tail in one kernel (stylenet/model.py:147-153, nn.LSTMCell nic/model.py:77):
//                      z = Wx[g*H+u, :] . x_g[r] + bx + Wh[g*H+u, :] . h[src[r]] + bh for the four gates of unit u
//                      (one warp per unit), gate nonlinearities, c' / h' written for row r; the beam re-ordering of the
//                      state (src_row, model.py:275-279) is a gather on READ, so no index_select kernels follow.
//   sn_decode_cell_groups : sn_decode_cell for up to 4 style groups of rows in one launch, each group with its own
//                      input weights (the collapsed chain of its style, model.py:115-155): the per-style sample() calls
//                      of one image (app/backend/model.py, one get_sample per style) become one beam search.
// fp32 weights and arithmetic in both precision modes (bf16 mode may be more accurate than it promises here).
#include "sn_common.cuh"

namespace {

constexpr int SK_WARPS = 8;
constexpr int SN_SKINNY_MAX_CHUNKS = 16;  // sn_skinny_linear: up to 16 x 16 rows
constexpr int SK_NR = 4;          // output features per warp

// The R input rows are NOT staged through shared memory: they are a few KB, every warp of the SM reads the same
// addresses, so they are L1 hits after the first touch -- a staging loop (dependent index -> row -> element loads, one
// element per thread and iteration) cost more than the whole contraction (27 us of a 57 us decode step, profiles/).
template <int RMAX>
__global__ void __launch_bounds__(SK_WARPS * 32, RMAX <= 8 ? 3 : 1) skinny_linear_kernel(
    const float* __restrict__ W, int64_t ldw, int N, int K, const float* __restrict__ X, int64_t ldx, int group_n,
    int group_x, const float* __restrict__ bias, float* __restrict__ out, int64_t ldo, int R,
    const int* __restrict__ x_rows, int rchunk) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int n0 = (blockIdx.x * SK_WARPS + warp) * SK_NR;
  if (n0 >= N) return;
  // grid.y = row chunk: this CTA handles rows [r0, r0 + R) of the caller's rows (one chunk, r0 = 0, when R <= 16)
  const int r0 = blockIdx.y * rchunk;
  R = min(R - r0, rchunk);
  // all SK_NR features of a warp lie in ONE x group (the host guarantees group_n % (SK_WARPS*SK_NR) == 0)
  const int xoff = group_n > 0 ? (n0 / group_n) * group_x : 0;
  const float* xr[RMAX];
#pragma unroll
  for (int r = 0; r < RMAX; ++r) xr[r] = X + (int64_t)(r < R ? (x_rows ? x_rows[r0 + r] : r0 + r) : 0) * ldx + xoff;
  float acc[RMAX][SK_NR];
#pragma unroll
  for (int r = 0; r < RMAX; ++r)
#pragma unroll
    for (int j = 0; j < SK_NR; ++j) acc[r][j] = 0.f;
  const bool vec = ((ldw & 3) == 0) && ((K & 3) == 0) && ((ldx & 3) == 0) && ((xoff & 3) == 0) &&
                   (((reinterpret_cast<uintptr_t>(W) | reinterpret_cast<uintptr_t>(X)) & 15) == 0);
  if (vec) {
#pragma unroll 2
    for (int k = lane * 4; k < K; k += 128) {
      float4 w[SK_NR];
#pragma unroll
      for (int j = 0; j < SK_NR; ++j)
        w[j] = (n0 + j < N) ? __ldg(reinterpret_cast<const float4*>(W + (int64_t)(n0 + j) * ldw + k)) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int r = 0; r < RMAX; ++r) {
        if (r < R) {
          const float4 x = __ldg(reinterpret_cast<const float4*>(xr[r] + k));
#pragma unroll
          for (int j = 0; j < SK_NR; ++j) acc[r][j] += w[j].x * x.x + w[j].y * x.y + w[j].z * x.z + w[j].w * x.w;
        }
      }
    }
  } else {
    for (int k = lane; k < K; k += 32) {
      float w[SK_NR];
#pragma unroll
      for (int j = 0; j < SK_NR; ++j) w[j] = (n0 + j < N) ? __ldg(W + (int64_t)(n0 + j) * ldw + k) : 0.f;
#pragma unroll
      for (int r = 0; r < RMAX; ++r)
        if (r < R) {
          const float x = __ldg(xr[r] + k);
#pragma unroll
          for (int j = 0; j < SK_NR; ++j) acc[r][j] += w[j] * x;
        }
    }
  }
#pragma unroll
  for (int r = 0; r < RMAX; ++r)
    if (r < R) {
#pragma unroll
      for (int j = 0; j < SK_NR; ++j) {
        const float s = sn::warp_sum(acc[r][j]);
        if (lane == 0 && n0 + j < N) out[(int64_t)(r0 + r) * ldo + n0 + j] = s + (bias ? bias[n0 + j] : 0.f);
      }
    }
}

// one warp per (unit, half): half 0 contracts the x part (Wx rows of the four gates), half 1 the recurrent part (W_hh
// rows); 4 units per CTA -> H/4 CTAs (128 at H = 512) instead of H/8
constexpr int DC_UNITS = SK_WARPS / 2;

// The cell of rows [r0, r0 + R) (R <= RMAX) for the units of this CTA.  Shared by sn_decode_cell (r0 = 0) and
// sn_decode_cell_groups (r0 = the row chunk of a style group): a row's arithmetic does not depend on r0 or RMAX.
template <int RMAX>
__device__ __forceinline__ void decode_cell_rows(
    int cell, int H, int r0, int R, const float* __restrict__ Wx, int64_t ldwx, int Kx, const float* __restrict__ X,
    int64_t ldx, int group_x, const float* __restrict__ bx, const float* __restrict__ Wh, const float* __restrict__ bh,
    const float* __restrict__ h_prev, const float* __restrict__ c_prev, const int* __restrict__ src_row,
    const int* __restrict__ x_rows, float* __restrict__ h_out, float* __restrict__ c_out) {
  __shared__ float zpart[DC_UNITS][2][RMAX][4];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int ul = warp >> 1, half = warp & 1;
  const int u = blockIdx.x * DC_UNITS + ul;
  float acc[RMAX][4];
#pragma unroll
  for (int r = 0; r < RMAX; ++r) acc[r][0] = acc[r][1] = acc[r][2] = acc[r][3] = 0.f;
  if (u < H) {
    if (half == 0) {
      // x part: row g*H+u of Wx against x group g (factored: U_g on a2_g ; LSTM: W_ih on x)
      const bool vec = ((ldwx & 3) == 0) && ((Kx & 3) == 0) && ((ldx & 3) == 0) && ((group_x & 3) == 0) &&
                       (((reinterpret_cast<uintptr_t>(Wx) | reinterpret_cast<uintptr_t>(X)) & 15) == 0);
      // (x_rows: row r of the input is X[x_rows[r]] -- the embedding lookup folded into the cell, collapsed chain)
      const float* xr[RMAX];
#pragma unroll
      for (int r = 0; r < RMAX; ++r) xr[r] = X + (int64_t)(r < R ? (x_rows ? x_rows[r0 + r] : r0 + r) : 0) * ldx;
      if (vec) {
#pragma unroll 2
        for (int k = lane * 4; k < Kx; k += 128) {
          float4 w[4];
#pragma unroll
          for (int g = 0; g < 4; ++g) w[g] = __ldg(reinterpret_cast<const float4*>(Wx + (int64_t)(g * H + u) * ldwx + k));
#pragma unroll
          for (int r = 0; r < RMAX; ++r)
            if (r < R) {
#pragma unroll
              for (int g = 0; g < 4; ++g) {
                const float4 x = __ldg(reinterpret_cast<const float4*>(xr[r] + g * group_x + k));
                acc[r][g] += w[g].x * x.x + w[g].y * x.y + w[g].z * x.z + w[g].w * x.w;
              }
            }
        }
      } else {
        for (int k = lane; k < Kx; k += 32) {
          float w[4];
#pragma unroll
          for (int g = 0; g < 4; ++g) w[g] = __ldg(Wx + (int64_t)(g * H + u) * ldwx + k);
#pragma unroll
          for (int r = 0; r < RMAX; ++r)
            if (r < R) {
#pragma unroll
              for (int g = 0; g < 4; ++g) acc[r][g] += w[g] * __ldg(xr[r] + g * group_x + k);
            }
        }
      }
    } else {
      // recurrent part: row g*H+u of W_hh against h_prev (rows gathered through src_row)
      const float* hr[RMAX];
#pragma unroll
      for (int r = 0; r < RMAX; ++r) hr[r] = h_prev + (int64_t)(r < R ? (src_row ? src_row[r0 + r] : r0 + r) : 0) * H;
      const bool vec = ((H & 3) == 0) && (((reinterpret_cast<uintptr_t>(Wh) | reinterpret_cast<uintptr_t>(h_prev)) & 15) == 0);
      if (vec) {
#pragma unroll 2
        for (int k = lane * 4; k < H; k += 128) {
          float4 w[4];
#pragma unroll
          for (int g = 0; g < 4; ++g) w[g] = __ldg(reinterpret_cast<const float4*>(Wh + (int64_t)(g * H + u) * H + k));
#pragma unroll
          for (int r = 0; r < RMAX; ++r)
            if (r < R) {
              const float4 x = __ldg(reinterpret_cast<const float4*>(hr[r] + k));
#pragma unroll
              for (int g = 0; g < 4; ++g) acc[r][g] += w[g].x * x.x + w[g].y * x.y + w[g].z * x.z + w[g].w * x.w;
            }
        }
      } else {
        for (int k = lane; k < H; k += 32) {
          float w[4];
#pragma unroll
          for (int g = 0; g < 4; ++g) w[g] = __ldg(Wh + (int64_t)(g * H + u) * H + k);
#pragma unroll
          for (int r = 0; r < RMAX; ++r)
            if (r < R) {
              const float x = __ldg(hr[r] + k);
#pragma unroll
              for (int g = 0; g < 4; ++g) acc[r][g] += w[g] * x;
            }
        }
      }
    }
#pragma unroll
    for (int r = 0; r < RMAX; ++r)
      if (r < R) {
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          const float s = sn::warp_sum(acc[r][g]);
          if (lane == 0) zpart[ul][half][r][g] = s;
        }
      }
  }
  __syncthreads();
  // finish: lane r of the x-part warp of a unit handles row r  (x part + bias_x first, then h part + bias_h: the order
  // of the two nn.Linear results in the reference, stylenet/model.py:147-150)
  if (u < H && half == 0 && lane < R) {
    const int r = r0 + lane;
    float z[4];
#pragma unroll
    for (int g = 0; g < 4; ++g)
      z[g] = (zpart[ul][0][lane][g] + (bx ? bx[g * H + u] : 0.f)) + (zpart[ul][1][lane][g] + (bh ? bh[g * H + u] : 0.f));
    const int sr = src_row ? src_row[r] : r;
    const float cp = c_prev[(int64_t)sr * H + u];
    const float zo = cell == SN_CELL_LSTM ? z[3] : z[2], zc = cell == SN_CELL_LSTM ? z[2] : z[3];
    const float gi = sn::sigmoidf_(z[0]), gf = sn::sigmoidf_(z[1]), go = sn::sigmoidf_(zo), gc = tanhf(zc);
    const float c = gf * cp + gi * gc;
    c_out[(int64_t)r * H + u] = c;
    h_out[(int64_t)r * H + u] = cell == SN_CELL_LSTM ? go * tanhf(c) : go * c;
  }
}

template <int RMAX>
__global__ void __launch_bounds__(SK_WARPS * 32) decode_cell_kernel(
    int cell, int H, int R, const float* __restrict__ Wx, int64_t ldwx, int Kx, const float* __restrict__ X, int64_t ldx,
    int group_x, const float* __restrict__ bx, const float* __restrict__ Wh, const float* __restrict__ bh,
    const float* __restrict__ h_prev, const float* __restrict__ c_prev, const int* __restrict__ src_row,
    const int* __restrict__ x_rows, float* __restrict__ h_out, float* __restrict__ c_out) {
  decode_cell_rows<RMAX>(cell, H, 0, R, Wx, ldwx, Kx, X, ldx, group_x, bx, Wh, bh, h_prev, c_prev, src_row, x_rows,
                         h_out, c_out);
}

// grid.y = (style group g, row chunk): group g owns rows [row_off[g], row_off[g+1]) and reads ITS input weights
// Wx + g*sWx / bx + g*sbx; W_hh, b_hh and the state are shared.  Chunks of <= `chunk` rows keep the RMAX <= 8 bodies
// (no spills); W_hh is re-read per chunk, from L2.
template <int RMAX>
__global__ void __launch_bounds__(SK_WARPS * 32, 1) decode_cell_groups_kernel(
    int cell, int H, const int* __restrict__ row_off, int chunk, int nchunk, const float* __restrict__ Wx,
    int64_t ldwx, int64_t sWx, int Kx, const float* __restrict__ X, int64_t ldx, int group_x,
    const float* __restrict__ bx, int64_t sbx, const float* __restrict__ Wh, const float* __restrict__ bh,
    const float* __restrict__ h_prev, const float* __restrict__ c_prev, const int* __restrict__ src_row,
    const int* __restrict__ x_rows, float* __restrict__ h_out, float* __restrict__ c_out) {
  const int g = blockIdx.y / nchunk;
  const int r0 = row_off[g] + (blockIdx.y % nchunk) * chunk;
  const int R = min(row_off[g + 1] - r0, chunk);
  if (R <= 0) return;                 // uniform over the CTA, before the body's barrier
  decode_cell_rows<RMAX>(cell, H, r0, R, Wx + g * sWx, ldwx, Kx, X, ldx, group_x, bx ? bx + g * sbx : nullptr, Wh, bh,
                         h_prev, c_prev, src_row, x_rows, h_out, c_out);
}

}  // namespace

extern "C" {

int32_t sn_skinny_max_rows(void) { return 16; }

int32_t sn_skinny_linear(const float* W, int64_t ldw, int64_t N, int64_t K, const float* X, int64_t ldx, int64_t R,
                         int64_t group_n, int64_t group_x, const float* bias, float* out, int64_t ldo,
                         const int32_t* x_rows, void* stream) {
  SN_REQUIRE(W && X && out && N > 0 && K > 0 && R > 0, "sn_skinny_linear: bad argument");
  SN_REQUIRE(R <= SN_SKINNY_MAX_CHUNKS * 16, "sn_skinny_linear: at most %d rows (got %lld); use sn_gemm",
             SN_SKINNY_MAX_CHUNKS * 16, (long long)R);
  SN_REQUIRE(group_n == 0 || group_n % (SK_WARPS * SK_NR) == 0, "sn_skinny_linear: group size must be a multiple of %d", SK_WARPS * SK_NR);
  const size_t smem = 0;
  // more than 16 rows (several styles of one image): balanced row chunks of <= 16 along grid.y, each one pass over W
  // (from L2 after the first chunk) on the spill-free RMAX = 16 body
  const int nchunk = (int)((R + 15) / 16);
  const int rchunk = (int)((R + nchunk - 1) / nchunk);
  const dim3 grid((unsigned)((N + SK_WARPS * SK_NR - 1) / (SK_WARPS * SK_NR)), (unsigned)nchunk);
  cudaStream_t st = (cudaStream_t)stream;
#define SN_SKINNY(RM) skinny_linear_kernel<RM><<<grid, SK_WARPS * 32, smem, st>>>(W, ldw, (int)N, (int)K, X, ldx, (int)group_n, (int)group_x, bias, out, ldo, (int)R, x_rows, rchunk)
  if (rchunk <= 4) SN_SKINNY(4);
  else if (rchunk == 5) SN_SKINNY(5);   // beam width 5, one image: the common single-image decode
  else if (rchunk <= 8) SN_SKINNY(8);
  else SN_SKINNY(16);
#undef SN_SKINNY
  return sn::check_launch("sn_skinny_linear");
}

int32_t sn_decode_cell(int32_t cell, int64_t H, int64_t R, const float* Wx, int64_t ldwx, int64_t Kx, const float* X,
                       int64_t ldx, int64_t group_x, const float* bx, const float* Wh, const float* bh,
                       const float* h_prev, const float* c_prev, const int32_t* src_row, const int32_t* x_rows,
                       float* h_out, float* c_out, void* stream) {
  SN_REQUIRE(cell == SN_CELL_FACTORED || cell == SN_CELL_LSTM, "sn_decode_cell: bad cell %d", cell);
  SN_REQUIRE(Wx && X && Wh && h_prev && c_prev && h_out && c_out && H > 0 && R > 0 && Kx > 0, "sn_decode_cell: bad argument");
  SN_REQUIRE(R <= 16, "sn_decode_cell: at most 16 rows (got %lld)", (long long)R);
  SN_REQUIRE(h_out != h_prev && c_out != c_prev, "sn_decode_cell: the state is gathered on read; in/out buffers must differ");
  const size_t smem = 0;
  const unsigned grid = (unsigned)((H + DC_UNITS - 1) / DC_UNITS);
  cudaStream_t st = (cudaStream_t)stream;
#define SN_CELL(RM) decode_cell_kernel<RM><<<grid, SK_WARPS * 32, smem, st>>>(cell, (int)H, (int)R, Wx, ldwx, (int)Kx, X, ldx, (int)group_x, bx, Wh, bh, h_prev, c_prev, src_row, x_rows, h_out, c_out)
  if (R <= 4) SN_CELL(4);
  else if (R == 5) SN_CELL(5);
  else if (R <= 8) SN_CELL(8);
  else SN_CELL(16);
#undef SN_CELL
  return sn::check_launch("sn_decode_cell");
}

int32_t sn_decode_cell_groups(int32_t cell, int64_t H, int64_t G, const int32_t* row_off, int64_t rows_max,
                              const float* Wx, int64_t ldwx, int64_t sWx, int64_t Kx, const float* X, int64_t ldx,
                              int64_t group_x, const float* bx, int64_t sbx, const float* Wh, const float* bh,
                              const float* h_prev, const float* c_prev, const int32_t* src_row, const int32_t* x_rows,
                              float* h_out, float* c_out, void* stream) {
  SN_REQUIRE(cell == SN_CELL_FACTORED || cell == SN_CELL_LSTM, "sn_decode_cell_groups: bad cell %d", cell);
  SN_REQUIRE(row_off && Wx && X && Wh && h_prev && c_prev && h_out && c_out && H > 0 && Kx > 0,
             "sn_decode_cell_groups: bad argument");
  SN_REQUIRE(G >= 1 && G <= 4, "sn_decode_cell_groups: 1..4 groups (got %lld)", (long long)G);
  SN_REQUIRE(rows_max >= 1 && rows_max <= 1024, "sn_decode_cell_groups: rows_max must be in 1..1024 (got %lld)",
             (long long)rows_max);
  SN_REQUIRE(h_out != h_prev && c_out != c_prev, "sn_decode_cell_groups: the state is gathered on read; in/out buffers must differ");
  const size_t smem = 0;
  const int nchunk = (int)((rows_max + 7) / 8);
  const int chunk = (int)((rows_max + nchunk - 1) / nchunk);
  const dim3 grid((unsigned)((H + DC_UNITS - 1) / DC_UNITS), (unsigned)(G * nchunk));
  cudaStream_t st = (cudaStream_t)stream;
#define SN_CELLG(RM) decode_cell_groups_kernel<RM><<<grid, SK_WARPS * 32, smem, st>>>(cell, (int)H, row_off, chunk, nchunk, Wx, ldwx, sWx, (int)Kx, X, ldx, (int)group_x, bx, sbx, Wh, bh, h_prev, c_prev, src_row, x_rows, h_out, c_out)
  if (chunk <= 4) SN_CELLG(4);
  else if (chunk == 5) SN_CELLG(5);     // beam width 5, one image per style: the multi-style serving request
  else SN_CELLG(8);
#undef SN_CELLG
  return sn::check_launch("sn_decode_cell_groups");
}

}  // extern "C"
