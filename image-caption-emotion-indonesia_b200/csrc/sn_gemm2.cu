// K2b: persistent CTA-pair GEMM on tcgen05 (cta_group::2) with pluggable epilogues.
//
//   D[M,N] = op(A) op(B)      bf16 operands, fp32 accumulation in TMEM, op in {NT, NN, TN}, 1..4 groups
//
// Why a second GEMM kernel: with CTA-private 128x128 tiles (sn_gemm_tc.cu) every 64-deep k-block needs 32 KB
// from L2 per 256 tensor-pipe cycles = 128 B/clk/SM, three times what L2 can deliver to all 148 SMs at once
// (~42 B/clk/SM) -> the tensor pipe saturates near 33 %.  A CTA pair computing one 256x256 tile with
// tcgen05.mma.cta_group::2 needs the same 32 KB per CTA per k-block but for 512 cycles of MMA work
// (64 B/clk/SM): twice the arithmetic intensity at the same shared-memory footprint.
//
// Structure (one cluster of 2 CTAs per SM pair, persistent over tiles, 576 threads per CTA):
//   warp 0      TMA producer (both CTAs): each CTA loads ITS 128 rows of A and ITS 128 rows of B of the k-block
//               into its own 5-stage ring (cp.async.bulk.tensor .cta_group::2), transaction bytes of both CTAs
//               complete on the LEADER's "full" mbarrier
//   warp 1      MMA issuer (leader CTA only): one lane issues 4 x tcgen05.mma.cta_group::2.kind::f16
//               (M=256, N=256, K=16) per stage; tcgen05.commit.multicast frees the stage in BOTH CTAs and, after
//               the last k-block, publishes the accumulator to BOTH CTAs' epilogue warps
//   warps 2..17 epilogue (both CTAs): 128 TMEM lanes x 256 columns per CTA; warp w reads lane quadrant w%4,
//               64-column slice (w-2)/4.  The accumulator is double-buffered in TMEM (2 x 256 columns) so the
//               epilogue of tile i runs under the MMAs of tile i+1.  tcgen05.ld hands every thread one ROW of
//               a 32x32 block; outputs go through a per-warp swizzled shared-memory transpose so that global
//               stores are 128-bit and row-contiguous (4 rows x 128 B per instruction) instead of 32 scattered
//               16-byte pieces (measured: LSU-throttled at ~1.5 TB/s before, see profiles/).
// Epilogues:
//   EPI_STORE   C fp32 and/or Cb bf16 (+bias, +beta*C)
//   EPI_PARTIAL split-K: raw fp32 partial tile into ws[split][M][N]; sn_gemm2_bf16 reduces them afterwards
//   EPI_STATS   vocabulary projection fused with log-softmax statistics: per (row, 64-column chunk) max, sum of
//               exp, arg-max; the target's logit.  Logits never leave the SM.
//   EPI_CELL_FWD / EPI_CELL_BWD  one time step of the recurrence for LARGE batches (K3 in the throughput regime): the
//               step's h_{t-1} W_hh^T (resp. dZ_{t+1} W_hh) GEMM with the LSTM / FactoredLSTM cell (resp. its
//               backward) fused into the epilogue -- see sn_recur_*_gemm below.
//   EPI_GRAD    recomputed logits -> (softmax - onehot) * scale written as the bf16 operand of the two backward
//               GEMMs, plus the count of logits above the target's (top-k accuracy).
#include <cuda.h>
#include <cuda_bf16.h>
#include <math.h>
#include <math_constants.h>

#include "sn_common.cuh"

namespace {

constexpr int BMC = 128;            // rows of A per CTA
constexpr int BM = 2 * BMC;         // tile rows per CTA pair
constexpr int BN = 256;             // default tile columns per CTA pair (each CTA stages half of them)
constexpr int BK = 64;
constexpr int UMMA_K = 16;
constexpr int A_BYTES = BMC * BK * 2;
constexpr int ACC_STAGES = 2;
constexpr int EPI_WARPS = 16;
constexpr int NTHREADS = 64 + 32 * EPI_WARPS;                    // 576
constexpr int XPOSE_BYTES = 32 * 32 * 4;                         // per-warp transpose buffer (32x32 fp32, swizzled)
// Tile geometry as a function of the pair tile width BN_ (256: the GEMMs; 128: the recurrence backward step, whose
// N = H = 512 would otherwise give too few tiles to occupy the SM pairs)
template <int BN_>
struct Geo {
  static constexpr int BNC = BN_ / 2;                            // rows of B staged per CTA
  static constexpr int B_BYTES = BNC * BK * 2;
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;          // 32 KB (BN 256) / 24 KB (BN 128) per CTA per stage
  static constexpr int STAGES = BN_ == 256 ? 5 : 6;
  static constexpr int TMEM_COLS = ACC_STAGES * BN_;             // 512 (the whole TMEM of the SM) / 256
  static constexpr int EPI_COLS = BN_ / (EPI_WARPS / 4);         // accumulator columns per epilogue warp: 64 / 32
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + EPI_WARPS * XPOSE_BYTES + 1024 + 256;
};

enum { EPI_STORE = 0, EPI_PARTIAL = 1, EPI_STATS = 2, EPI_GRAD = 3, EPI_CELL_FWD = 4, EPI_CELL_BWD = 5,
       EPI_GRADW = 6 /* EPI_GRAD with per-row weights */ };

struct TmaSet { CUtensorMap m[4]; };

struct G2Args {
  int M, N, K;
  int groups, splits;
  int a_mn_major, b_mn_major;
  // EPI_STORE / EPI_PARTIAL
  float* C; __nv_bfloat16* Cb; int64_t ldc, ldcb;
  const float* bias; float beta;
  int64_t strideC, strideCb, strideBias;
  float* ws;                       // split-K partials [groups*splits][M][N]
  // EPI_STATS / EPI_GRAD (vocabulary projection: rows = tokens, columns = vocabulary)
  const int64_t* targets;
  float* pmax; float* psum; int32_t* pidx; int nchunks;   // [M, nchunks]
  float* tlogit;                   // [M] logit of the target column
  const float* lse;                // [M]
  float scale, scale_log2;
  __nv_bfloat16* dL; int64_t lddl; // [M, lddl] gradient w.r.t. the logits
  int32_t* above;                  // [M] number of logits strictly above the target's
  // EPI_CELL_FWD / EPI_CELL_BWD (one recurrence step; rows = samples of the step, all row-indexed pointers are
  // already offset to the step's first packed row)
  int cell, Hdim;
  const float* xp; const float* bhh; const float* c_prev;      // [M,4H], [4H], [M,H] (NULL = zeros)
  float* h_out; __nv_bfloat16* hb_out; float* c_out; float* gates_out;
  const float* gates_in; const float* c_cur; const float* dh_in; float* dc_carry;   // bwd: [M,4H], [M,H], [M,H], [M,H]
  float* dz_out; __nv_bfloat16* dzb_out;                        // bwd: [M,4H] fp32 (optional) and bf16
  const float* row_weight;         // EPI_GRADW: [M] per-row gradient weight
};

// EPI_GRADW: the one-hot term of a weighted row, |w| * scale
__device__ __forceinline__ float wscale(const G2Args& g, int64_t row) { return fabsf(__ldg(g.row_weight + row)) * g.scale; }

// ---- PTX wrappers ------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
// address of the same shared-memory variable in CTA `rank` of the cluster (shared::cluster window)
__device__ __forceinline__ uint32_t mapa(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void cluster_sync() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_bar) {
  // default semantics (.release.cta): the hand-off only orders this warp's tcgen05.ld (already waited for) before the
  // MMA issuer's next tcgen05.mma, which tcgen05.fence::before/after_thread_sync covers; a cluster-scope release
  // would drain every outstanding global store of the warp first (MEMBAR.ALL + ERRBAR, ~20 % of the epilogue).
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "G2_WAIT_LOOP:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra G2_WAIT_DONE;\n\t"
      "bra G2_WAIT_LOOP;\n\t"
      "G2_WAIT_DONE:\n\t}" ::"r"(bar), "r"(parity) : "memory");
}
// consumer-side wait with cluster-scope acquire (the barrier is completed by the peer CTA's arrivals)
__device__ __forceinline__ void mbar_wait_cluster(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "G2_WAITC_LOOP:\n\t"
      "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra G2_WAITC_DONE;\n\t"
      "bra G2_WAITC_LOOP;\n\t"
      "G2_WAITC_DONE:\n\t}" ::"r"(bar), "r"(parity) : "memory");
}
// both CTAs of the pair load into their own shared memory; the bytes complete on the leader's barrier
__device__ __forceinline__ void tma_load_2d_2sm(uint32_t dst, const CUtensorMap* map, uint32_t leader_bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(map), "r"(leader_bar), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tmem_alloc2(uint32_t dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(ncols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc2(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void umma2_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc) : "memory");
}
// arrive on the barrier at this shared-memory offset in BOTH CTAs once all prior MMAs have retired
__device__ __forceinline__ void umma2_commit_mc(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(bar), "h"((uint16_t)3) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// issue the TMEM load (32 lanes x 32 columns, one row per thread); results are valid after tmem_ld_wait(r)
__device__ __forceinline__ void tmem_ld32_issue(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr) : "memory");
}
// the registers are in/out operands so that no use of r[] can be scheduled above the wait
__device__ __forceinline__ void tmem_ld_wait(uint32_t (&r)[32]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
      : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]),
        "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15]),
        "+r"(r[16]), "+r"(r[17]), "+r"(r[18]), "+r"(r[19]), "+r"(r[20]), "+r"(r[21]), "+r"(r[22]), "+r"(r[23]),
        "+r"(r[24]), "+r"(r[25]), "+r"(r[26]), "+r"(r[27]), "+r"(r[28]), "+r"(r[29]), "+r"(r[30]), "+r"(r[31])
      :: "memory");
}
__device__ __forceinline__ float ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
constexpr float LOG2E = 1.4426950408889634f;
__device__ __forceinline__ float fast_sigmoid(float x) {
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(1.0f + ex2(-LOG2E * x)));
  return r;
}
__device__ __forceinline__ float fast_tanh(float x) {
  float y;
  asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

// ---- per-warp 32x32 fp32 transpose through shared memory -------------------------------------------------------
// write side: thread = row, 8 x STS.128; element (row, c) lives at row*32 + ((c/4) ^ (row & 7))*4 + c%4 -> the 8 rows of
// a quarter-warp hit 8 different 16-byte bank groups.  read side: lane -> (row 4i + lane/8, columns 4*(lane%8)..+3),
// LDS.128, again conflict-free; a warp-level global store then covers 4 rows x 128 contiguous bytes.
__device__ __forceinline__ void xpose_write(float* buf, int lane, const float (&v)[32]) {
#pragma unroll
  for (int c4 = 0; c4 < 8; ++c4)
    *reinterpret_cast<float4*>(buf + lane * 32 + ((c4 ^ (lane & 7)) << 2)) =
        make_float4(v[4 * c4], v[4 * c4 + 1], v[4 * c4 + 2], v[4 * c4 + 3]);
}
__device__ __forceinline__ float4 xpose_read(const float* buf, int lane, int i) {
  const int row = 4 * i + (lane >> 3), c4 = lane & 7;
  return *reinterpret_cast<const float4*>(buf + row * 32 + ((c4 ^ (row & 7)) << 2));
}

// shared-memory matrix descriptor: start>>4 [0,14), LBO>>4 [16,30), SBO>>4 [32,46), version=1 [46,48),
// layout_type [61,64) = 2 (SWIZZLE_128B)
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}

// bf16 output of a 32x32 block held one ROW per thread: pack to bf16x2, transpose through 2 KB of shared memory
// (16-byte units, unit u of row r at r*64 + (u ^ ((r>>1)&3))*16: conflict-free both ways), then 4 x STG.128 where
// every instruction covers 8 rows x 64 contiguous bytes.  Requires ld % 8 == 0 and a 16-byte aligned base for the
// vector path; ragged right edges fall back to scalar stores.
__device__ __forceinline__ void store_block_bf16(float* xbuf, int lane, const float (&v)[32], __nv_bfloat16* base,
                                                 int64_t ld, int row0, int M, int nb, int ncols, bool vec_ok) {
  uint8_t* buf = reinterpret_cast<uint8_t*>(xbuf);
  __syncwarp();
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    __nv_bfloat162 p0 = __floats2bfloat162_rn(v[8 * u], v[8 * u + 1]), p1 = __floats2bfloat162_rn(v[8 * u + 2], v[8 * u + 3]);
    __nv_bfloat162 p2 = __floats2bfloat162_rn(v[8 * u + 4], v[8 * u + 5]), p3 = __floats2bfloat162_rn(v[8 * u + 6], v[8 * u + 7]);
    uint4 pk;
    pk.x = *reinterpret_cast<uint32_t*>(&p0); pk.y = *reinterpret_cast<uint32_t*>(&p1);
    pk.z = *reinterpret_cast<uint32_t*>(&p2); pk.w = *reinterpret_cast<uint32_t*>(&p3);
    *reinterpret_cast<uint4*>(buf + lane * 64 + ((u ^ ((lane >> 1) & 3)) << 4)) = pk;
  }
  __syncwarp();
  const int u = lane & 3;
  const int n8 = nb + 8 * u;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int r = 8 * i + (lane >> 2);
    const uint4 pk = *reinterpret_cast<const uint4*>(buf + r * 64 + ((u ^ ((r >> 1) & 3)) << 4));
    const int rr = row0 + r;
    if (rr >= M || n8 >= ncols) continue;
    __nv_bfloat16* dst = base + (int64_t)rr * ld + n8;
    if (vec_ok && n8 + 8 <= ncols) {
      *reinterpret_cast<uint4*>(dst) = pk;
    } else {
      const __nv_bfloat16* e = reinterpret_cast<const __nv_bfloat16*>(&pk);
#pragma unroll
      for (int k = 0; k < 8; ++k)
        if (n8 + k < ncols) dst[k] = e[k];
    }
  }
}

struct Tile { int m0, n0, grp, split, kb0, nkb; };

__device__ __forceinline__ Tile decode_tile(const G2Args& g, int tile, int tiles_m, int tiles_n, int total_kb, int bn) {
  // Tile order: the fastest-varying index walks the SMALLER operand, so the ~74 tiles in flight share a few tiles of
  // the larger operand (read from HBM once) while the smaller one stays L2-resident (M >> N: all n-tiles of an
  // m-tile run side by side; measured before: A re-fetched from HBM behind the streaming output writes).
  Tile t;
  int mt, nt, rest;
  if (g.M > g.N) {
    nt = tile % tiles_n; rest = tile / tiles_n;
    mt = rest % tiles_m; rest /= tiles_m;
  } else {
    mt = tile % tiles_m; rest = tile / tiles_m;
    nt = rest % tiles_n; rest /= tiles_n;
  }
  t.split = rest % g.splits;
  t.grp = rest / g.splits;
  t.m0 = mt * BM;
  t.n0 = nt * bn;
  if (g.splits == 1) {
    t.kb0 = 0; t.nkb = total_kb;
  } else {
    t.kb0 = (total_kb * t.split) / g.splits;
    t.nkb = (total_kb * (t.split + 1)) / g.splits - t.kb0;
  }
  return t;
}


template <int EPI, int BN_>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(NTHREADS, 1)   // 18 warps (allocated as 20) x 96 registers
gemm2_kernel(const __grid_constant__ TmaSet tma_a, const __grid_constant__ TmaSet tma_b, const G2Args g) {
  constexpr int BNC = Geo<BN_>::BNC, B_BYTES = Geo<BN_>::B_BYTES, STAGE_BYTES = Geo<BN_>::STAGE_BYTES;
  constexpr int STAGES = Geo<BN_>::STAGES, TMEM_COLS = Geo<BN_>::TMEM_COLS, EPI_COLS = Geo<BN_>::EPI_COLS;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  float* xpose0 = reinterpret_cast<float*>(smem + STAGES * STAGE_BYTES);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + STAGES * STAGE_BYTES + EPI_WARPS * XPOSE_BYTES);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 2 * ACC_STAGES);
  const uint32_t smem_base = smem_u32(smem);
  const uint32_t full0 = smem_u32(bars), empty0 = smem_u32(bars + STAGES);
  const uint32_t tfull0 = smem_u32(bars + 2 * STAGES), tempty0 = smem_u32(bars + 2 * STAGES + ACC_STAGES);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int pair = blockIdx.x >> 1, npairs = gridDim.x >> 1;
  const int tiles_m = (g.M + BM - 1) / BM, tiles_n = (g.N + BN_ - 1) / BN_;
  const int total_tiles = tiles_m * tiles_n * g.groups * g.splits;
  const int total_kb = (g.K + BK - 1) / BK;

  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; ++s) { mbar_init(full0 + 8 * s, 1); mbar_init(empty0 + 8 * s, 1); }
    for (int s = 0; s < ACC_STAGES; ++s) { mbar_init(tfull0 + 8 * s, 1); mbar_init(tempty0 + 8 * s, 2 * EPI_WARPS); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0 && lane == 0) {
    for (int i = 0; i < g.groups; ++i) {
      asm volatile("prefetch.tensormap [%0];" ::"l"(&tma_a.m[i]) : "memory");
      asm volatile("prefetch.tensormap [%0];" ::"l"(&tma_b.m[i]) : "memory");
    }
  }
  if (warp == 1) tmem_alloc2(smem_u32(tmem_slot), TMEM_COLS);
  tc_fence_before();
  cluster_sync();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===================== TMA producer (both CTAs) =====================
    if (lane == 0) {
      int s = 0;
      uint32_t ph = 0;
      for (int tile = pair; tile < total_tiles; tile += npairs) {
        const Tile t = decode_tile(g, tile, tiles_m, tiles_n, total_kb, BN_);
        const CUtensorMap* map_a = &tma_a.m[t.grp];
        const CUtensorMap* map_b = &tma_b.m[t.grp];
        const int m0 = t.m0 + (int)rank * BMC, n0 = t.n0 + (int)rank * BNC;
        int k0 = t.kb0 * BK;
        for (int kb = 0; kb < t.nkb; ++kb, k0 += BK) {
          mbar_wait(empty0 + 8 * s, ph ^ 1);
          const uint32_t sa = smem_base + s * STAGE_BYTES, sb = sa + A_BYTES;
          const uint32_t lbar = mapa(full0 + 8 * s, 0);
          if (rank == 0) mbar_expect_tx(full0 + 8 * s, 2 * STAGE_BYTES);
          if (!g.a_mn_major) {
            tma_load_2d_2sm(sa, map_a, lbar, k0, m0);                    // box {64 k, 128 rows}
          } else {
            tma_load_2d_2sm(sa, map_a, lbar, m0, k0);                    // box {64 m, 64 k-rows}
            tma_load_2d_2sm(sa + A_BYTES / 2, map_a, lbar, m0 + 64, k0);
          }
          if (!g.b_mn_major) {
            tma_load_2d_2sm(sb, map_b, lbar, k0, n0);
          } else {
            tma_load_2d_2sm(sb, map_b, lbar, n0, k0);
            if (BNC == 128) tma_load_2d_2sm(sb + B_BYTES / 2, map_b, lbar, n0 + 64, k0);
          }
          if (++s == STAGES) { s = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (leader CTA, ONE thread) =====================
    // The whole issue loop runs in a single thread and is kept to a handful of instructions per MMA (descriptors are
    // a 64-bit add on a per-stage base): at 135 tensor-pipe cycles per 256x256x16 MMA a ~100-instruction issue path
    // per k-block was itself the bottleneck (ncu: the issuing warp never waited on a barrier, profiles/r1_i).
    if (rank == 0 && lane == 0) {
      // instruction descriptor: D=f32 [4,6)=1, A=bf16 [7,10)=1, B=bf16 [10,13)=1, a_major bit15, b_major bit16,
      // N>>3 [17,23), M>>4 [24,29)
      const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)g.a_mn_major << 15) |
                             ((uint32_t)g.b_mn_major << 16) | ((uint32_t)(BN_ >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
      // K-major: advance 32 B inside the 128 B swizzle row; SBO = 1024 B between 8-row groups.
      // MN-major: advance two 8-k-row groups (2 KB); LBO = 8 KB between the two 64-wide MN chunks.
      const uint64_t adesc0 = g.a_mn_major ? make_desc(smem_base, A_BYTES / 2, 1024) : make_desc(smem_base, 16, 1024);
      const uint64_t bdesc0 = g.b_mn_major ? make_desc(smem_base + A_BYTES, BNC == 128 ? B_BYTES / 2 : 16, 1024)
                                           : make_desc(smem_base + A_BYTES, 16, 1024);
      const uint64_t astep = (g.a_mn_major ? 2048 : 32) >> 4, bstep = (g.b_mn_major ? 2048 : 32) >> 4;
      int s = 0, as = 0;
      uint32_t ph = 0, aph = 0;
      for (int tile = pair; tile < total_tiles; tile += npairs) {
        const Tile t = decode_tile(g, tile, tiles_m, tiles_n, total_kb, BN_);
        mbar_wait_cluster(tempty0 + 8 * as, aph ^ 1);      // epilogues of both CTAs drained this accumulator
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + (uint32_t)(as * BN_);
        for (int kb = 0; kb < t.nkb; ++kb) {
          mbar_wait(full0 + 8 * s, ph);
          tc_fence_after();
          const uint64_t ad = adesc0 + (uint64_t)(s * (STAGE_BYTES >> 4)), bd = bdesc0 + (uint64_t)(s * (STAGE_BYTES >> 4));
          umma2_bf16(tmem_d, ad, bd, idesc, kb ? 1u : 0u);
#pragma unroll
          for (int k = 1; k < BK / UMMA_K; ++k) umma2_bf16(tmem_d, ad + k * astep, bd + k * bstep, idesc, 1u);
          umma2_commit_mc(empty0 + 8 * s);
          if (kb == t.nkb - 1) umma2_commit_mc(tfull0 + 8 * as);
          if (++s == STAGES) { s = 0; ph ^= 1; }
        }
        if (++as == ACC_STAGES) { as = 0; aph ^= 1; }
      }
    }
    __syncwarp();
  } else {
    // ===================== epilogue (warps 2..17, both CTAs) =====================
    const int q = warp & 3;                      // TMEM lane quadrant of this warp
    const int slice = (warp - 2) >> 2;           // 64-column slice of the 256-wide accumulator
    float* xbuf = xpose0 + (warp - 2) * (XPOSE_BYTES / 4);
    const uint32_t tempty_leader0 = mapa(tempty0, 0);
    int acc_it = 0;
    for (int tile = pair; tile < total_tiles; tile += npairs, ++acc_it) {
      const Tile t = decode_tile(g, tile, tiles_m, tiles_n, total_kb, BN_);
      const int as = acc_it & 1;
      const uint32_t aph = (acc_it >> 1) & 1;
      if (EPI == EPI_CELL_FWD || EPI == EPI_CELL_BWD) {
        // The cell epilogues are memory-bound and their operands do not depend on the accumulator: pull this warp's
        // rows of XP / c / gates / dh into L2 now, while the MMAs of the tile are still running (the warp would
        // otherwise just wait on the barrier below and then pay the full DRAM latency twice per tile).
        const int H = g.Hdim;
        const int prow0 = t.m0 + (int)rank * BMC + q * 32;
        if (EPI == EPI_CELL_FWD) {
          const int U0 = t.n0 >> 2;
          for (int idx = lane; idx < 80; idx += 32) {
            const int ph = idx / 40, rem = idx - ph * 40, k = rem / 5, a = rem - k * 5;
            const int rr = prow0 + slice * 8 + k;
            const float* p = a < 4 ? g.xp + (int64_t)rr * 4 * H + a * H + U0 + 32 * ph
                                   : (g.c_prev ? g.c_prev + (int64_t)rr * H + U0 + 32 * ph : nullptr);
            if (rr < g.M && p) prefetch_l2(p);
          }
        } else {
          const int u0 = t.n0 + slice * EPI_COLS;
          for (int idx = lane; idx < 32 * 8; idx += 32) {
            const int rr = prow0 + (idx >> 3), a = idx & 7;
            const float* p = a < 4 ? g.gates_in + (int64_t)rr * 4 * H + a * H + u0
                           : a == 4 ? g.c_cur + (int64_t)rr * H + u0
                           : a == 5 ? (g.c_prev ? g.c_prev + (int64_t)rr * H + u0 : nullptr)
                           : a == 6 ? g.dh_in + (int64_t)rr * H + u0 : g.dc_carry + (int64_t)rr * H + u0;
            if (rr < g.M && u0 < g.N && p) prefetch_l2(p);
          }
        }
      }
      mbar_wait(tfull0 + 8 * as, aph);
      tc_fence_after();
      const int row0 = t.m0 + (int)rank * BMC + q * 32;     // first row of this warp's 32-row band
      const int row = row0 + lane;                          // the row this thread holds after tcgen05.ld
      const int ncol0 = t.n0 + slice * EPI_COLS;
      const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(as * BN_ + slice * EPI_COLS);
      const bool row_ok = row < g.M;

      if (EPI == EPI_STORE || EPI == EPI_PARTIAL) {
        float* Cg = nullptr;
        __nv_bfloat16* Cbg = nullptr;
        const float* bias = nullptr;
        int64_t ldc = g.ldc;
        float beta = 0.f;
        if (EPI == EPI_PARTIAL) {
          Cg = g.ws + (int64_t)(t.grp * g.splits + t.split) * g.M * g.N;
          ldc = g.N;
        } else {
          Cg = g.C ? g.C + t.grp * g.strideC : nullptr;
          Cbg = g.Cb ? g.Cb + t.grp * g.strideCb : nullptr;
          bias = g.bias ? g.bias + t.grp * g.strideBias : nullptr;
          beta = g.beta;
        }
        const bool vec_c = Cg && ((ldc & 3) == 0) && ((reinterpret_cast<uintptr_t>(Cg) & 15) == 0);
        const bool vec_cb = Cbg && ((g.ldcb & 3) == 0) && ((reinterpret_cast<uintptr_t>(Cbg) & 7) == 0);
        const bool bf16_only = (EPI == EPI_STORE) && !Cg && Cbg && ((g.ldcb & 7) == 0) &&
                               ((reinterpret_cast<uintptr_t>(Cbg) & 15) == 0);
#pragma unroll 1
        for (int c0 = 0; c0 < EPI_COLS; c0 += 32) {
          uint32_t r[32];
          tmem_ld32_issue(taddr + c0, r);
          const int nb = ncol0 + c0;
          if (bf16_only) {
            // bf16-only output (activations of the forward chain): bias in the row layout, packed transpose
            float v[32];
            if (bias && nb + 32 <= g.N && ((reinterpret_cast<uintptr_t>(bias + nb) & 15) == 0)) {
#pragma unroll
              for (int j = 0; j < 32; j += 4) {
                const float4 b = __ldg(reinterpret_cast<const float4*>(bias + nb + j));
                v[j] = b.x; v[j + 1] = b.y; v[j + 2] = b.z; v[j + 3] = b.w;
              }
            } else {
#pragma unroll
              for (int j = 0; j < 32; ++j) v[j] = (bias && nb + j < g.N) ? __ldg(bias + nb + j) : 0.f;
            }
            tmem_ld_wait(r);
            if (nb >= g.N || row0 >= g.M) continue;                   // warp-uniform
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] += __uint_as_float(r[j]);
            store_block_bf16(xbuf, lane, v, Cbg, g.ldcb, row0, g.M, nb, g.N, true);
            continue;
          }
          const int n4 = nb + 4 * (lane & 7);              // this lane's 4 columns in the store phase
          float4 b4 = make_float4(0.f, 0.f, 0.f, 0.f);
          if (bias && nb < g.N) {
            if (n4 + 4 <= g.N && ((reinterpret_cast<uintptr_t>(bias + n4) & 15) == 0)) {
              b4 = __ldg(reinterpret_cast<const float4*>(bias + n4));
            } else {
              if (n4 < g.N) b4.x = __ldg(bias + n4);
              if (n4 + 1 < g.N) b4.y = __ldg(bias + n4 + 1);
              if (n4 + 2 < g.N) b4.z = __ldg(bias + n4 + 2);
              if (n4 + 3 < g.N) b4.w = __ldg(bias + n4 + 3);
            }
          }
          tmem_ld_wait(r);
          if (nb >= g.N || row0 >= g.M) continue;                     // warp-uniform
          float v[32];
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]);
          __syncwarp();
          xpose_write(xbuf, lane, v);
          __syncwarp();
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const int rr = row0 + 4 * i + (lane >> 3);
            float4 x = xpose_read(xbuf, lane, i);
            if (rr >= g.M || n4 >= g.N) continue;
            x.x += b4.x; x.y += b4.y; x.z += b4.z; x.w += b4.w;
            const bool full = n4 + 4 <= g.N;
            if (Cg) {
              float* dst = Cg + (int64_t)rr * ldc + n4;
              if (full && vec_c) {
                if (EPI == EPI_STORE && beta != 0.f) {
                  const float4 o = *reinterpret_cast<const float4*>(dst);
                  x.x += beta * o.x; x.y += beta * o.y; x.z += beta * o.z; x.w += beta * o.w;
                }
                *reinterpret_cast<float4*>(dst) = x;
              } else {
                float e[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
                for (int k = 0; k < 4; ++k)
                  if (n4 + k < g.N) {
                    if (EPI == EPI_STORE && beta != 0.f) e[k] += beta * dst[k];
                    dst[k] = e[k];
                  }
                x = make_float4(e[0], e[1], e[2], e[3]);
              }
            }
            if (Cbg) {
              __nv_bfloat16* dstb = Cbg + (int64_t)rr * g.ldcb + n4;
              if (full && vec_cb) {
                __nv_bfloat162 p0 = __floats2bfloat162_rn(x.x, x.y), p1 = __floats2bfloat162_rn(x.z, x.w);
                uint2 pk;
                pk.x = *reinterpret_cast<uint32_t*>(&p0); pk.y = *reinterpret_cast<uint32_t*>(&p1);
                *reinterpret_cast<uint2*>(dstb) = pk;
              } else {
                const float e[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
                for (int k = 0; k < 4; ++k)
                  if (n4 + k < g.N) dstb[k] = __float2bfloat16(e[k]);
              }
            }
          }
        }
      } else if (EPI == EPI_STATS) {
        // online max / sum-exp / arg-max over this warp's 64 columns (two 32-column halves; the
        // partials are per (row, 64-column chunk)); one thread = one token row
        const int64_t tgt = row_ok ? g.targets[row] : -1;
        float mx = -CUDART_INF_F, se = 0.f;
        int mi = 0x7fffffff;
#pragma unroll 1
        for (int c0 = 0; c0 < EPI_COLS; c0 += 32) {
          uint32_t r[32];
          tmem_ld32_issue(taddr + c0, r);
          const int nb = ncol0 + c0;
          float v[32];
          if (nb + 32 <= g.N && ((reinterpret_cast<uintptr_t>(g.bias + nb) & 15) == 0)) {
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
              const float4 b = __ldg(reinterpret_cast<const float4*>(g.bias + nb + j));
              v[j] = b.x; v[j + 1] = b.y; v[j + 2] = b.z; v[j + 3] = b.w;
            }
          } else {
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] = (nb + j < g.N) ? __ldg(g.bias + nb + j) : -CUDART_INF_F;
          }
          tmem_ld_wait(r);
          if (!row_ok || nb >= g.N) continue;
          float cm4[4] = {-CUDART_INF_F, -CUDART_INF_F, -CUDART_INF_F, -CUDART_INF_F};
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            v[j] += __uint_as_float(r[j]);                 // columns >= N stay -inf
            cm4[j & 3] = fmaxf(cm4[j & 3], v[j]);
          }
          const float cm = fmaxf(fmaxf(cm4[0], cm4[1]), fmaxf(cm4[2], cm4[3]));
          if (cm > mx) {
            // first (lowest) column attaining the new maximum
            int first = 0;
#pragma unroll
            for (int j = 31; j >= 0; --j) if (v[j] == cm) first = j;
            mi = nb + first;
            se *= ex2((mx - cm) * LOG2E);
            mx = cm;
          }
          const float mb = mx * LOG2E;
          float s4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
          for (int j = 0; j < 32; ++j) s4[j & 3] += ex2(fmaf(v[j], LOG2E, -mb));
          se += (s4[0] + s4[1]) + (s4[2] + s4[3]);
          if (tgt >= nb && tgt < nb + 32) {
#pragma unroll
            for (int j = 0; j < 32; ++j) if (nb + j == (int)tgt) g.tlogit[row] = v[j];
          }
        }
        if (row_ok && ncol0 < g.N) {
          const int64_t o = (int64_t)row * g.nchunks + (ncol0 / EPI_COLS);
          g.pmax[o] = mx; g.psum[o] = se; g.pidx[o] = mi;
        }
      } else if (EPI == EPI_CELL_FWD) {
        // Columns are GATE-INTERLEAVED 64 units at a time (sn_cast_bf16_gate_interleave): the 256-column tile holds the
        // four gate pre-activations of units U0..U0+63, one gate per 64-column slice = per epilogue warp of a lane
        // quadrant.  The four warps of a quadrant (same 32 rows) exchange their gates through shared memory, 32 units
        // per phase, then each warp finishes 8 of the 32 rows with lane = unit: every global access of the cell update
        // (XP, c, h, gates) is a full 128-byte row segment.  (One row per thread, as tcgen05.ld delivers the data,
        // costs 32 cache lines per instruction and was LSU-bound at 3x the HBM time.)
        const int H = g.Hdim;
        const bool lstm = g.cell == SN_CELL_LSTM;
        float* qbuf = xpose0 + q * (4 * 32 * 32);          // [4 gates][32 rows][32 units], swizzled rows
        const int bar_id = 1 + q;
        const int U0 = t.n0 >> 2;                            // first unit of this tile
#pragma unroll 1
        for (int ph = 0; ph < 2; ++ph) {
          uint32_t r[32];
          tmem_ld32_issue(taddr + 32 * ph, r);
          tmem_ld_wait(r);
          if (ph == 1) {      // accumulator fully read: hand the TMEM stage back before the memory-bound part
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_cluster(tempty_leader0 + 8 * as);
          }
          {
            float v[32];
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]);
            xpose_write(qbuf + slice * 1024, lane, v);       // gate `slice`, row = lane
          }
          asm volatile("bar.sync %0, 128;" ::"r"(bar_id) : "memory");
          const int unit = U0 + 32 * ph + lane;
          float bh[4];
#pragma unroll
          for (int k = 0; k < 4; ++k) bh[k] = g.bhh ? __ldg(g.bhh + k * H + unit) : 0.f;
          const int sw = lane >> 2, lo = lane & 3;
#pragma unroll 8
          for (int k = 0; k < 8; ++k) {
            const int rl = slice * 8 + k;                    // row inside the quadrant
            const int rr = row0 + rl;
            if (rr >= g.M) continue;
            const float* xp = g.xp + (int64_t)rr * 4 * H + unit;
            const int so = rl * 32 + ((sw ^ (rl & 7)) << 2) + lo;
            const float z0 = qbuf[so] + __ldg(xp) + bh[0];
            const float z1 = qbuf[1024 + so] + __ldg(xp + H) + bh[1];
            const float z2 = qbuf[2048 + so] + __ldg(xp + 2 * H) + bh[2];
            const float z3 = qbuf[3072 + so] + __ldg(xp + 3 * H) + bh[3];
            const float cp = g.c_prev ? __ldg(g.c_prev + (int64_t)rr * H + unit) : 0.f;
            // gate blocks: FactoredLSTM (i, f, o, c~), h = o*c ; LSTM (i, f, g, o), h = o*tanh(c)
            const float gi = fast_sigmoid(z0), gf = fast_sigmoid(z1);
            const float g2 = lstm ? fast_tanh(z2) : fast_sigmoid(z2);
            const float g3 = lstm ? fast_sigmoid(z3) : fast_tanh(z3);
            const float go = lstm ? g3 : g2, gc = lstm ? g2 : g3;
            const float c = gf * cp + gi * gc;
            const float h = lstm ? go * fast_tanh(c) : go * c;
            g.hb_out[(int64_t)rr * H + unit] = __float2bfloat16(h);
            if (g.h_out) g.h_out[(int64_t)rr * H + unit] = h;
            if (g.c_out) g.c_out[(int64_t)rr * H + unit] = c;
            if (g.gates_out) {
              float* gp = g.gates_out + (int64_t)rr * 4 * H + unit;
              gp[0] = gi; gp[H] = gf; gp[2 * H] = g2; gp[3 * H] = g3;
            }
          }
          asm volatile("bar.sync %0, 128;" ::"r"(bar_id) : "memory");
        }
        continue;                                            // TMEM stage already released above
      } else if (EPI == EPI_CELL_BWD) {
        // accumulator = dh_rec[row, unit] = dZ_{t+1} W_hh.  Transposed through shared memory so that a lane holds 4
        // consecutive units of a row: all loads / stores of the cell backward are float4 and row-contiguous
        // (4 rows x 128 B per instruction).
        const int H = g.Hdim;
        const bool lstm = g.cell == SN_CELL_LSTM;
#pragma unroll 1
        for (int c0 = 0; c0 < EPI_COLS; c0 += 32) {
          uint32_t r[32];
          tmem_ld32_issue(taddr + c0, r);
          tmem_ld_wait(r);
          if (row0 >= g.M || ncol0 + c0 >= g.N) continue;       // warp-uniform
          {
            float v[32];
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]);
            __syncwarp();
            xpose_write(xbuf, lane, v);
            __syncwarp();
          }
          const int u4 = ncol0 + c0 + 4 * (lane & 7);
#pragma unroll 2
          for (int i = 0; i < 8; ++i) {
            const int rr = row0 + 4 * i + (lane >> 3);
            const float4 acc4 = xpose_read(xbuf, lane, i);
            if (rr >= g.M) continue;
            const float* gp = g.gates_in + (int64_t)rr * 4 * H + u4;
            const float4 g0 = *reinterpret_cast<const float4*>(gp), g1 = *reinterpret_cast<const float4*>(gp + H);
            const float4 g2 = *reinterpret_cast<const float4*>(gp + 2 * H), g3 = *reinterpret_cast<const float4*>(gp + 3 * H);
            const float4 cc4 = *reinterpret_cast<const float4*>(g.c_cur + (int64_t)rr * H + u4);
            const float4 cp4 = g.c_prev ? *reinterpret_cast<const float4*>(g.c_prev + (int64_t)rr * H + u4)
                                        : make_float4(0.f, 0.f, 0.f, 0.f);
            const float4 dh4 = *reinterpret_cast<const float4*>(g.dh_in + (int64_t)rr * H + u4);
            float4 dcar4 = *reinterpret_cast<const float4*>(g.dc_carry + (int64_t)rr * H + u4);
            const float acc[4] = {acc4.x, acc4.y, acc4.z, acc4.w};
            const float gt0[4] = {g0.x, g0.y, g0.z, g0.w}, gt1[4] = {g1.x, g1.y, g1.z, g1.w};
            const float gt2[4] = {g2.x, g2.y, g2.z, g2.w}, gt3[4] = {g3.x, g3.y, g3.z, g3.w};
            const float cc[4] = {cc4.x, cc4.y, cc4.z, cc4.w}, cp[4] = {cp4.x, cp4.y, cp4.z, cp4.w};
            const float dh[4] = {dh4.x, dh4.y, dh4.z, dh4.w};
            float dcar[4] = {dcar4.x, dcar4.y, dcar4.z, dcar4.w};
            float zz[4][4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const float dht = dh[e] + acc[e];
              const float gi = gt0[e], gf = gt1[e];
              const float go = lstm ? gt3[e] : gt2[e], gc = lstm ? gt2[e] : gt3[e];
              float d_o, dc;
              if (lstm) {
                const float tc = fast_tanh(cc[e]);
                d_o = dht * tc;
                dc = dcar[e] + dht * go * (1.f - tc * tc);
              } else {
                d_o = dht * cc[e];
                dc = dcar[e] + dht * go;
              }
              const float di = dc * gc, df = dc * cp[e], dg = dc * gi;
              dcar[e] = dc * gf;
              const float zi = di * gi * (1.f - gi), zf = df * gf * (1.f - gf);
              const float zo = d_o * go * (1.f - go), zc = dg * (1.f - gc * gc);
              zz[0][e] = zi; zz[1][e] = zf;
              zz[2][e] = lstm ? zc : zo; zz[3][e] = lstm ? zo : zc;
            }
            *reinterpret_cast<float4*>(g.dc_carry + (int64_t)rr * H + u4) = make_float4(dcar[0], dcar[1], dcar[2], dcar[3]);
#pragma unroll
            for (int qq = 0; qq < 4; ++qq) {
              if (g.dz_out)
                *reinterpret_cast<float4*>(g.dz_out + (int64_t)rr * 4 * H + qq * H + u4) =
                    make_float4(zz[qq][0], zz[qq][1], zz[qq][2], zz[qq][3]);
              __nv_bfloat162 p0 = __floats2bfloat162_rn(zz[qq][0], zz[qq][1]), p1 = __floats2bfloat162_rn(zz[qq][2], zz[qq][3]);
              uint2 pk;
              pk.x = *reinterpret_cast<uint32_t*>(&p0); pk.y = *reinterpret_cast<uint32_t*>(&p1);
              *reinterpret_cast<uint2*>(g.dzb_out + (int64_t)rr * 4 * H + qq * H + u4) = pk;
            }
          }
        }
      } else {  // EPI_GRAD, EPI_GRADW
        constexpr bool kW = EPI == EPI_GRADW;
        const int64_t tgt = row_ok ? g.targets[row] : -1;
        // a row weight w scales the row's gradient: log2(|w| scale) joins the exponent offset, the one-hot term is
        // |w| scale, and the sign is applied last (w = 0: exp2(-inf) = 0, so the row is zeros)
        // (a separate instantiation, so the unweighted epilogue keeps its registers; the weighted one reads w (L1) where
        // it is used instead of holding |w| scale and the sign across the loop, which spilled at the 96-register cap)
        const float escale = row_ok ? (kW ? g.scale_log2 + log2f(fabsf(__ldg(g.row_weight + row))) : g.scale_log2) -
                                          g.lse[row] * LOG2E
                                    : 0.f;   // exp2 argument offset: -lse + log(scale); w = 1 adds an exact 0
        const float tl = row_ok ? g.tlogit[row] : 0.f;
        int cnt = 0;
#pragma unroll 1
        for (int c0 = 0; c0 < EPI_COLS; c0 += 32) {
          uint32_t r[32];
          tmem_ld32_issue(taddr + c0, r);
          const int nb = ncol0 + c0;
          float v[32];
          if (nb + 32 <= g.N && ((reinterpret_cast<uintptr_t>(g.bias + nb) & 15) == 0)) {
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
              const float4 b = __ldg(reinterpret_cast<const float4*>(g.bias + nb + j));
              v[j] = b.x; v[j + 1] = b.y; v[j + 2] = b.z; v[j + 3] = b.w;
            }
          } else {
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] = (nb + j < g.N) ? __ldg(g.bias + nb + j) : 0.f;
          }
          tmem_ld_wait(r);
          if (nb >= g.lddl || row0 >= g.M) continue;                  // warp-uniform
          if (nb + 32 <= g.N) {
            // (softmax - onehot) * scale with the scale folded into the exponent: 5 instructions per logit
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              const float x = v[j] + __uint_as_float(r[j]);
              cnt += (x > tl);
              v[j] = ex2(fmaf(x, LOG2E, escale));
            }
            if (tgt >= nb && tgt < nb + 32) {
#pragma unroll
              for (int j = 0; j < 32; ++j) if (nb + j == (int)tgt) v[j] -= kW ? wscale(g, row) : g.scale;
            }
            if (!row_ok) {
              cnt = 0;
#pragma unroll
              for (int j = 0; j < 32; ++j) v[j] = 0.f;
            }
          } else {
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              const int n = nb + j;
              const float x = v[j] + __uint_as_float(r[j]);
              const bool in = row_ok && n < g.N;
              cnt += (in && x > tl);
              const float p = ex2(fmaf(x, LOG2E, escale));
              // zeros = K padding of the next GEMMs
              v[j] = in ? p - (n == (int)tgt ? (kW ? wscale(g, row) : g.scale) : 0.f) : 0.f;
            }
          }
          if (kW && row_ok && __ldg(g.row_weight + row) < 0.f) {
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] = -v[j];
          }
          if (g.dL) store_block_bf16(xbuf, lane, v, g.dL, g.lddl, row0, g.M, nb, (int)g.lddl, true);
        }
        if (g.above && cnt) atomicAdd(g.above + row, cnt);
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(tempty_leader0 + 8 * as);
    }
  }
  tc_fence_before();
  cluster_sync();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc2(tmem_base, TMEM_COLS);
  }
}

// ---- split-K reduction: out = sum_s ws[s] (+bias) (+beta*C) ------------------------------------------------
__global__ void __launch_bounds__(256) splitk_reduce_kernel(const float* __restrict__ ws, int splits, int64_t M, int64_t N,
                                                            float* C, int64_t ldc, __nv_bfloat16* Cb, int64_t ldcb,
                                                            const float* __restrict__ bias, float beta) {
  const int64_t total4 = M * N / 4;        // N % 4 == 0 (checked by the host)
  const int64_t MN = M * N;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total4; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t e = i * 4;
    const int64_t m = e / N, n = e - m * N;
    float4 a = *reinterpret_cast<const float4*>(ws + e);
    for (int s = 1; s < splits; ++s) {
      const float4 b = *reinterpret_cast<const float4*>(ws + s * MN + e);
      a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w;
    }
    if (bias) { a.x += bias[n]; a.y += bias[n + 1]; a.z += bias[n + 2]; a.w += bias[n + 3]; }
    if (C) {
      float* dst = C + m * ldc + n;
      if (beta != 0.f) { a.x += beta * dst[0]; a.y += beta * dst[1]; a.z += beta * dst[2]; a.w += beta * dst[3]; }
      dst[0] = a.x; dst[1] = a.y; dst[2] = a.z; dst[3] = a.w;
    }
    if (Cb) {
      __nv_bfloat16* d = Cb + m * ldcb + n;
      d[0] = __float2bfloat16(a.x); d[1] = __float2bfloat16(a.y); d[2] = __float2bfloat16(a.z); d[3] = __float2bfloat16(a.w);
    }
  }
}

// ---- vocabulary statistics: combine the per-chunk partials of one row ------------------------------------------
// lse = log sum exp(logits); row_loss = lse - logit[target]; argmax = lowest index of the maximum (torch.max);
// above[row] is zeroed for the gradient / ranking pass.  One warp per row.
__global__ void __launch_bounds__(256) vocab_combine_kernel(const float* __restrict__ pmax, const float* __restrict__ psum,
                                                            const int32_t* __restrict__ pidx, int nchunks, int64_t N,
                                                            const float* __restrict__ tlogit, float* __restrict__ lse,
                                                            float* __restrict__ row_loss, int64_t* __restrict__ argmax,
                                                            int32_t* __restrict__ above) {
  const int lane = threadIdx.x & 31;
  const int64_t row = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (row >= N) return;
  float mx = -CUDART_INF_F;
  int mi = 0x7fffffff;
  for (int c = lane; c < nchunks; c += 32) {
    const float v = pmax[row * nchunks + c];
    const int i = pidx[row * nchunks + c];
    if (v > mx || (v == mx && i < mi)) { mx = v; mi = i; }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ov = __shfl_xor_sync(0xffffffffu, mx, o);
    const int oi = __shfl_xor_sync(0xffffffffu, mi, o);
    if (ov > mx || (ov == mx && oi < mi)) { mx = ov; mi = oi; }
  }
  float s = 0.f;
  for (int c = lane; c < nchunks; c += 32) s += psum[row * nchunks + c] * expf(pmax[row * nchunks + c] - mx);
  s = sn::warp_sum(s);
  if (lane == 0) {
    const float l = mx + logf(s);
    lse[row] = l;
    if (row_loss) row_loss[row] = l - tlogit[row];
    if (argmax) argmax[row] = mi;
    if (above) above[row] = 0;
  }
}

__global__ void rank_hit_kernel(const int32_t* __restrict__ above, int64_t N, int32_t k, int32_t* __restrict__ hit) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < N) hit[i] = above[i] < k ? 1 : 0;
}

// ---- host side -------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                             const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                             CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeFn get_encode() {
  static EncodeFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeFn>(p);
  }
  return fn;
}

int32_t encode_2d(CUtensorMap* map, const void* base, int64_t inner, int64_t rows, int64_t pitch_elems, int box_inner,
                  int box_rows) {
  EncodeFn enc = get_encode();
  if (!enc) return sn::fail(-4, "cuTensorMapEncodeTiled entry point not available");
  cuuint64_t dims[2] = {(cuuint64_t)inner, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)pitch_elems * 2};
  cuuint32_t box[2] = {(cuuint32_t)box_inner, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return sn::fail(-5, "cuTensorMapEncodeTiled failed (%d): base=%p inner=%lld rows=%lld pitch=%lld", (int)r,
                                         base, (long long)inner, (long long)rows, (long long)pitch_elems);
  return 0;
}

// a_rows: valid rows of a K-major A (rows beyond are zero-filled by TMA; default M)
int32_t make_maps(int32_t op, int64_t M, int64_t N, int64_t K, const void* A, int64_t lda, const void* B, int64_t ldb,
                  int32_t batch, int64_t strideA, int64_t strideB, TmaSet& ta, TmaSet& tb, G2Args& g, int64_t a_rows = -1, int bn = BN) {
  if (a_rows < 0) a_rows = M;
  g.a_mn_major = (op == SN_OP_TN) ? 1 : 0;
  g.b_mn_major = (op == SN_OP_NT) ? 0 : 1;
  const __nv_bfloat16* Ab = (const __nv_bfloat16*)A;
  const __nv_bfloat16* Bb = (const __nv_bfloat16*)B;
  for (int i = 0; i < 4; ++i) {
    int gi = i < batch ? i : 0;
    int32_t rc;
    if (!g.a_mn_major) rc = encode_2d(&ta.m[i], Ab + gi * strideA, K, a_rows, lda, BK, BMC);     // A[M,K]
    else rc = encode_2d(&ta.m[i], Ab + gi * strideA, M, K, lda, 64, BK);                      // A stored [K,M]
    if (rc) return rc;
    if (!g.b_mn_major) rc = encode_2d(&tb.m[i], Bb + gi * strideB, K, N, ldb, BK, bn / 2);  // B[N,K]
    else rc = encode_2d(&tb.m[i], Bb + gi * strideB, N, K, ldb, 64, BK);                      // B stored [K,N]
    if (rc) return rc;
  }
  return 0;
}

template <int EPI, int BN_ = BN>
int32_t launch(const TmaSet& ta, const TmaSet& tb, const G2Args& g, cudaStream_t st, const char* what, int max_pairs = 0) {
  static thread_local bool configured = false;
  if (!configured) {
    SN_CUDA(cudaFuncSetAttribute(gemm2_kernel<EPI, BN_>, cudaFuncAttributeMaxDynamicSharedMemorySize, Geo<BN_>::SMEM_BYTES));
    configured = true;
  }
  const int64_t tiles = (int64_t)((g.M + BM - 1) / BM) * ((g.N + BN_ - 1) / BN_) * g.groups * g.splits;
  int64_t pairs = sn::dev_info().sm_count / 2;
  if (max_pairs > 0 && max_pairs < pairs) pairs = max_pairs;     // leave SMs to kernels on other streams
  if (tiles < pairs) pairs = tiles;
  gemm2_kernel<EPI, BN_><<<(unsigned)(2 * pairs), NTHREADS, Geo<BN_>::SMEM_BYTES, st>>>(ta, tb, g);
  return sn::check_launch(what);
}

int32_t check_operands(const char* what, const void* A, int64_t lda, const void* B, int64_t ldb, int64_t strideA,
                       int64_t strideB) {
  SN_REQUIRE(A && B, "%s: null operand", what);
  SN_REQUIRE((lda % 8) == 0 && (ldb % 8) == 0 && (strideA % 8) == 0 && (strideB % 8) == 0,
             "%s: bf16 leading dimensions / group strides must be multiples of 8 elements (TMA 16-byte rule): "
             "lda=%lld ldb=%lld", what, (long long)lda, (long long)ldb);
  SN_REQUIRE(((uintptr_t)A & 15) == 0 && ((uintptr_t)B & 15) == 0, "%s: operands must be 16-byte aligned", what);
  return 0;
}

}  // namespace

extern "C" int64_t sn_gemm2_ws_bytes(int64_t M, int64_t N, int32_t batch, int32_t splits) {
  if (splits <= 1) return 0;
  return (int64_t)sizeof(float) * M * N * batch * splits;
}

extern "C" int32_t sn_gemm2_bf16(int32_t op, int64_t M, int64_t N, int64_t K, const void* A, int64_t lda, const void* B,
                                 int64_t ldb, float* C, int64_t ldc, void* Cb, int64_t ldcb, const float* bias, float beta,
                                 int32_t batch, int64_t strideA, int64_t strideB, int64_t strideC, int64_t strideCb,
                                 int64_t strideBias, int32_t splits, void* ws, int64_t ws_bytes, int32_t max_pairs,
                                 void* stream) {
  SN_REQUIRE(op >= 0 && op <= 2, "sn_gemm2_bf16: bad op %d", op);
  SN_REQUIRE(batch >= 1 && batch <= 4, "sn_gemm2_bf16: 1..4 groups supported, got %d", batch);
  SN_REQUIRE(M >= 0 && N >= 0 && K > 0, "sn_gemm2_bf16: bad dims");
  if (M == 0 || N == 0) return 0;
  SN_REQUIRE(C || Cb, "sn_gemm2_bf16: no output");
  int32_t rc = check_operands("sn_gemm2_bf16", A, lda, B, ldb, strideA, strideB);
  if (rc) return rc;
  const int64_t total_kb = (K + BK - 1) / BK;
  if (splits < 1) splits = 1;
  if (splits > total_kb) splits = (int32_t)total_kb;
  TmaSet ta, tb;
  G2Args g = {};
  g.M = (int)M; g.N = (int)N; g.K = (int)K; g.groups = batch; g.splits = splits;
  rc = make_maps(op, M, N, K, A, lda, B, ldb, batch, strideA, strideB, ta, tb, g);
  if (rc) return rc;
  g.C = C; g.Cb = (__nv_bfloat16*)Cb; g.ldc = ldc; g.ldcb = ldcb; g.bias = bias; g.beta = beta;
  g.strideC = strideC; g.strideCb = strideCb; g.strideBias = strideBias;
  cudaStream_t st = (cudaStream_t)stream;
  if (splits == 1) return launch<EPI_STORE>(ta, tb, g, st, "sn_gemm2_bf16", max_pairs);
  SN_REQUIRE((N % 4) == 0, "sn_gemm2_bf16: split-K needs N %% 4 == 0");
  SN_REQUIRE(ws && ws_bytes >= sn_gemm2_ws_bytes(M, N, batch, splits), "sn_gemm2_bf16: split-K work space too small");
  SN_REQUIRE(((uintptr_t)ws & 15) == 0, "sn_gemm2_bf16: work space must be 16-byte aligned");
  g.ws = (float*)ws;
  rc = launch<EPI_PARTIAL>(ta, tb, g, st, "sn_gemm2_bf16(split-K)", max_pairs);
  if (rc) return rc;
  for (int gi = 0; gi < batch; ++gi) {
    int64_t blocks = (M * N / 4 + 255) / 256;
    int64_t cap = (int64_t)sn::dev_info().sm_count * 8;
    if (blocks > cap) blocks = cap;
    splitk_reduce_kernel<<<(unsigned)blocks, 256, 0, st>>>(
        g.ws + (int64_t)gi * splits * M * N, splits, M, N, C ? C + gi * strideC : nullptr, ldc,
        Cb ? (__nv_bfloat16*)Cb + gi * strideCb : nullptr, ldcb, bias ? bias + gi * strideBias : nullptr, beta);
    rc = sn::check_launch("sn_gemm2_bf16(reduce)");
    if (rc) return rc;
  }
  return 0;
}

extern "C" int64_t sn_vocab_ws_bytes(int64_t N, int64_t V) {
  const int64_t nchunks = (V + 63) / 64;
  return N * nchunks * 12;       // pmax, psum (fp32) + pidx (int32)
}

extern "C" int32_t sn_vocab_nll_fwd(int64_t N, int64_t V, int64_t H, const void* Hb, int64_t ldh, const void* Wb,
                                    int64_t ldw, const float* bias, const int64_t* targets, void* ws, int64_t ws_bytes,
                                    float* tlogit, float* lse, float* row_loss, int64_t* argmax, int32_t* above,
                                    void* stream) {
  SN_REQUIRE(N >= 0 && V > 0 && H > 0, "sn_vocab_nll_fwd: bad dims");
  if (N == 0) return 0;
  SN_REQUIRE(bias && targets && tlogit && lse, "sn_vocab_nll_fwd: null argument");
  SN_REQUIRE(ws && ws_bytes >= sn_vocab_ws_bytes(N, V), "sn_vocab_nll_fwd: work space too small");
  int32_t rc = check_operands("sn_vocab_nll_fwd", Hb, ldh, Wb, ldw, 0, 0);
  if (rc) return rc;
  const int nchunks = (int)((V + 63) / 64);
  TmaSet ta, tb;
  G2Args g = {};
  g.M = (int)N; g.N = (int)V; g.K = (int)H; g.groups = 1; g.splits = 1;
  rc = make_maps(SN_OP_NT, N, V, H, Hb, ldh, Wb, ldw, 1, 0, 0, ta, tb, g);
  if (rc) return rc;
  g.bias = bias; g.targets = targets; g.nchunks = nchunks;
  g.pmax = (float*)ws; g.psum = g.pmax + N * nchunks; g.pidx = (int32_t*)(g.psum + N * nchunks);
  g.tlogit = tlogit;
  cudaStream_t st = (cudaStream_t)stream;
  rc = launch<EPI_STATS>(ta, tb, g, st, "sn_vocab_nll_fwd");
  if (rc) return rc;
  vocab_combine_kernel<<<(unsigned)((N + 7) / 8), 256, 0, st>>>(g.pmax, g.psum, g.pidx, nchunks, N, tlogit, lse, row_loss,
                                                               argmax, above);
  return sn::check_launch("sn_vocab_nll_fwd(combine)");
}

extern "C" int32_t sn_vocab_nll_bwd(int64_t N, int64_t V, int64_t H, const void* Hb, int64_t ldh, const void* Wb,
                                    int64_t ldw, const float* bias, const int64_t* targets, const float* tlogit,
                                    const float* lse, float grad_scale, const float* row_weight, void* dL,
                                    int64_t lddl, int32_t* above, int32_t* top5hit, void* stream) {
  SN_REQUIRE(N >= 0 && V > 0 && H > 0, "sn_vocab_nll_bwd: bad dims");
  if (N == 0) return 0;
  SN_REQUIRE(bias && targets && tlogit && lse, "sn_vocab_nll_bwd: null argument");
  SN_REQUIRE(!dL || (lddl >= V && (lddl % 8) == 0 && ((uintptr_t)dL & 15) == 0),
             "sn_vocab_nll_bwd: dL pitch must be >= V, a multiple of 8, base 16-byte aligned");
  SN_REQUIRE(!top5hit || above, "sn_vocab_nll_bwd: top5hit needs the `above` counter");
  int32_t rc = check_operands("sn_vocab_nll_bwd", Hb, ldh, Wb, ldw, 0, 0);
  if (rc) return rc;
  TmaSet ta, tb;
  G2Args g = {};
  g.M = (int)N; g.N = (int)V; g.K = (int)H; g.groups = 1; g.splits = 1;
  rc = make_maps(SN_OP_NT, N, V, H, Hb, ldh, Wb, ldw, 1, 0, 0, ta, tb, g);
  if (rc) return rc;
  g.bias = bias; g.targets = targets; g.tlogit = (float*)tlogit; g.lse = lse; g.scale = grad_scale; g.scale_log2 = log2f(grad_scale);
  g.row_weight = row_weight;
  g.dL = (__nv_bfloat16*)dL; g.lddl = dL ? lddl : V; g.above = above;
  cudaStream_t st = (cudaStream_t)stream;
  rc = row_weight ? launch<EPI_GRADW>(ta, tb, g, st, "sn_vocab_nll_bwd") : launch<EPI_GRAD>(ta, tb, g, st, "sn_vocab_nll_bwd");
  if (rc) return rc;
  if (top5hit) {
    rank_hit_kernel<<<(unsigned)((N + 255) / 256), 256, 0, st>>>(above, N, 5, top5hit);
    return sn::check_launch("sn_vocab_nll_bwd(top5)");
  }
  return 0;
}

// ---- K3, large-batch form: one tcgen05 GEMM per time step with the cell fused into the epilogue ------------------
namespace {

// Wp[ublk*256 + q*64 + uu, :] = bf16(W[q*H + ublk*64 + uu, :])  (rows of the four gate blocks interleaved 64 units at a
// time: a 256-column accumulator tile = all four gates of 64 units, one gate per epilogue warp of a lane quadrant)
__global__ void gate_interleave_kernel(const float* __restrict__ W, int64_t H, int64_t K, int64_t ldw,
                                       __nv_bfloat16* __restrict__ Wp, int64_t ldp) {
  const int64_t total = 4 * H * ldp;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t n = i / ldp, k = i - n * ldp;
    const int64_t ublk = n >> 8, q = (n >> 6) & 3, uu = n & 63;
    const int64_t src_row = q * H + ublk * 64 + uu;
    Wp[n * ldp + k] = __float2bfloat16(k < K ? W[src_row * ldw + k] : 0.f);
  }
}

// Hprevb[row(b,t), :] = Hb[row(b,t-1), :] (zeros at t = 0): the h_{t-1} operand of dW_hh = dZ^T Hprev
__global__ void hprev_gather_kernel(const __nv_bfloat16* __restrict__ Hb, const int32_t* __restrict__ row_b,
                                    const int32_t* __restrict__ row_t, const int32_t* __restrict__ off, int64_t N,
                                    int64_t H, __nv_bfloat16* __restrict__ Hprevb) {
  const int64_t per_row = H >> 3;                      // 16-byte pieces
  const int64_t total = N * per_row;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / per_row, c = (i - r * per_row) << 3;
    const int t = row_t[r];
    uint4 v = make_uint4(0u, 0u, 0u, 0u);
    if (t > 0) v = *reinterpret_cast<const uint4*>(Hb + ((int64_t)off[t - 1] + row_b[r]) * H + c);
    *reinterpret_cast<uint4*>(Hprevb + r * H + c) = v;
  }
}

}  // namespace

extern "C" int32_t sn_cast_bf16_gate_interleave(const float* W, int64_t H, int64_t K, int64_t ldw, void* Wp, int64_t ldp,
                                                void* stream) {
  SN_REQUIRE(W && Wp && H > 0 && (H % 64) == 0 && K > 0 && ldw >= K && ldp >= K && (ldp % 8) == 0,
             "sn_cast_bf16_gate_interleave: bad arguments");
  int64_t blocks = (4 * H * ldp + 255) / 256;
  int64_t cap = (int64_t)sn::dev_info().sm_count * 16;
  if (blocks > cap) blocks = cap;
  gate_interleave_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(W, H, K, ldw, (__nv_bfloat16*)Wp, ldp);
  return sn::check_launch("sn_cast_bf16_gate_interleave");
}

extern "C" int32_t sn_recur_fwd_gemm(int32_t cell, int64_t H, int64_t B, const int32_t* bs_host, const int32_t* off_host,
                                     int32_t T, const float* XP, const void* Wp_bf16, const float* bhh, float* Hall,
                                     void* Hb, float* Call, float* gates, const void* zeros_bf16, void* stream) {
  SN_REQUIRE(cell == SN_CELL_FACTORED || cell == SN_CELL_LSTM, "sn_recur_fwd_gemm: bad cell %d", cell);
  SN_REQUIRE(H > 0 && (H % 64) == 0 && B > 0 && T > 0, "sn_recur_fwd_gemm: hidden size must be a multiple of 64");
  SN_REQUIRE(bs_host && off_host && XP && Wp_bf16 && Hb && Call && zeros_bf16, "sn_recur_fwd_gemm: null argument");
  int32_t rc = check_operands("sn_recur_fwd_gemm", Hb, H, Wp_bf16, H, 0, 0);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  __nv_bfloat16* Hbb = (__nv_bfloat16*)Hb;
  for (int t = 0; t < T; ++t) {
    const int64_t M = bs_host[t], r0 = off_host[t];
    if (M <= 0) break;
    TmaSet ta, tb;
    G2Args g = {};
    g.M = (int)M; g.N = (int)(4 * H); g.K = (int)H; g.groups = 1; g.splits = 1;
    // A = h_{t-1} rows of the samples still alive (zeros before the first step)
    const void* A = t == 0 ? zeros_bf16 : (const void*)(Hbb + (int64_t)off_host[t - 1] * H);
    rc = make_maps(SN_OP_NT, M, 4 * H, H, A, H, Wp_bf16, H, 1, 0, 0, ta, tb, g);
    if (rc) return rc;
    g.cell = cell; g.Hdim = (int)H;
    g.xp = XP + r0 * 4 * H; g.bhh = bhh;
    g.c_prev = t == 0 ? nullptr : Call + (int64_t)off_host[t - 1] * H;
    g.h_out = Hall ? Hall + r0 * H : nullptr; g.hb_out = Hbb + r0 * H;
    g.c_out = Call + r0 * H; g.gates_out = gates ? gates + r0 * 4 * H : nullptr;
    rc = launch<EPI_CELL_FWD>(ta, tb, g, st, "sn_recur_fwd_gemm");
    if (rc) return rc;
  }
  return 0;
}

extern "C" int32_t sn_recur_hprev(const void* Hb, const int32_t* row_b, const int32_t* row_t, const int32_t* offsets,
                                  int64_t N, int64_t H, void* Hprevb, void* stream) {
  SN_REQUIRE(Hb && row_b && row_t && offsets && Hprevb && N >= 0 && H > 0 && (H % 8) == 0, "sn_recur_hprev: bad arguments");
  if (N == 0) return 0;
  int64_t blocks = (N * (H >> 3) + 255) / 256;
  int64_t cap = (int64_t)sn::dev_info().sm_count * 16;
  if (blocks > cap) blocks = cap;
  hprev_gather_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>((const __nv_bfloat16*)Hb, row_b, row_t, offsets, N, H,
                                                                          (__nv_bfloat16*)Hprevb);
  return sn::check_launch("sn_recur_hprev");
}

extern "C" int32_t sn_recur_bwd_gemm(int32_t cell, int64_t H, int64_t B, const int32_t* bs_host, const int32_t* off_host,
                                     int32_t T, const void* Whh_bf16, const float* Call, const float* gates,
                                     const float* dHall, float* dZ, void* dZb, float* dc_carry, const void* zeros_bf16,
                                     void* stream) {
  SN_REQUIRE(cell == SN_CELL_FACTORED || cell == SN_CELL_LSTM, "sn_recur_bwd_gemm: bad cell %d", cell);
  SN_REQUIRE(H > 0 && (H % 64) == 0 && B > 0 && T > 0, "sn_recur_bwd_gemm: hidden size must be a multiple of 64");
  SN_REQUIRE(bs_host && off_host && Whh_bf16 && Call && gates && dHall && dZb && dc_carry && zeros_bf16,
             "sn_recur_bwd_gemm: null argument");
  int32_t rc = check_operands("sn_recur_bwd_gemm", dZb, 4 * H, Whh_bf16, H, 0, 0);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  SN_CUDA(cudaMemsetAsync(dc_carry, 0, sizeof(float) * (size_t)B * (size_t)H, st));
  __nv_bfloat16* dZbb = (__nv_bfloat16*)dZb;
  for (int t = T - 1; t >= 0; --t) {
    const int64_t M = bs_host[t], r0 = off_host[t];
    if (M <= 0) continue;
    const int64_t Mnext = (t + 1 < T) ? bs_host[t + 1] : 0;
    TmaSet ta, tb;
    G2Args g = {};
    g.M = (int)M; g.N = (int)H; g.K = (int)(4 * H); g.groups = 1; g.splits = 1;
    // A = dZ_{t+1} rows of the samples alive at t+1; the other samples of step t (and all of the last step) read
    // zeros: rows past the tensor map's extent are zero-filled by TMA
    const void* A = Mnext > 0 ? (const void*)(dZbb + (int64_t)off_host[t + 1] * 4 * H) : zeros_bf16;
    rc = make_maps(SN_OP_NN, M, H, 4 * H, A, 4 * H, Whh_bf16, H, 1, 0, 0, ta, tb, g, Mnext > 0 ? Mnext : 1, 128);
    if (rc) return rc;
    g.cell = cell; g.Hdim = (int)H;
    g.gates_in = gates + r0 * 4 * H; g.c_cur = Call + r0 * H;
    g.c_prev = t == 0 ? nullptr : Call + (int64_t)off_host[t - 1] * H;
    g.dh_in = dHall + r0 * H; g.dc_carry = dc_carry;
    g.dz_out = dZ ? dZ + r0 * 4 * H : nullptr; g.dzb_out = dZbb + r0 * 4 * H;
    rc = launch<EPI_CELL_BWD, 128>(ta, tb, g, st, "sn_recur_bwd_gemm");
    if (rc) return rc;
  }
  return 0;
}
