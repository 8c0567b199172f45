/*
 * sn100.h -- C ABI of libsn100.so: hand-written sm_100a CUDA for the StyleNet / NIC caption-decoder
 * hot path (SURVEY.md section 8).  This is the drop-in boundary below the PyTorch module surface:
 * plain pointers and sizes only, no torch / ATen / pybind types.
 *
 * The reference (deryrahman/image-caption-emotion-indonesia) has NO native code and no FFI: every
 * function below replaces a *library call site* that the reference makes through torch eager.  The
 * reference call site each entry point replaces is cited as `file:line` (paths relative to the
 * reference repository root).  INTEGRATION.md shows the reference-side binding (ctypes).
 *
 * Conventions (SURVEY.md section 8b)
 *   - every function returns int32: 0 ok; <0 argument/shape/alignment error detected before launch
 *     (text via sn_last_error()); >0 a cudaError_t from the launch.  No exceptions, no exit().
 *   - all pointers are DEVICE pointers owned by the caller (PyTorch caching allocator); the library
 *     never allocates, frees or retains them.  Work space is caller-provided.
 *   - row-major everywhere; activations are time-major packed [N, *] (N = sum of lengths; row of
 *     (sample b, step t) = off[t] + b, off[t] = sum_{s<t} batch_sizes[s]); weights keep the
 *     nn.Linear layout [out, in].
 *   - kernels are launched on the `stream` argument (cudaStream_t passed as void*), asynchronously.
 *   - no CPU fallback: a device that is not sm_100 is a hard error.
 */
#ifndef SN100_H_
#define SN100_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SN_VERSION 100

/* GEMM operand layouts */
#define SN_OP_NT 0 /* C[M,N] = A[M,K] * B[N,K]^T   (y = x W^T, nn.Linear forward)            */
#define SN_OP_NN 1 /* C[M,N] = A[M,K] * B[K,N]     (dx = dy W)                                */
#define SN_OP_TN 2 /* C[M,N] = A[K,M]^T * B[K,N]   (dW = dy^T x)                              */

/* GEMM arithmetic */
#define SN_PREC_F32 0   /* fp32 FFMA, exact-fp32 accumulation (fp32 parity mode, <=1e-5)       */
#define SN_PREC_BF16X6 1 /* fp32-grade accuracy on the bf16 tensor cores: 3 bf16 limbs per operand, 6 limb products laid
                            out along K (sn_split_limbs_* + sn_gemm2_bf16 / sn_gemm_bf16); fp32 mode's large GEMMs  */
#define SN_PREC_BF16 2  /* tcgen05 kind::f16 bf16 operands, fp32 accumulate in TMEM            */

/* recurrent cell kinds */
#define SN_CELL_FACTORED 0 /* gate blocks (i,f,o,c~); h = o*c        stylenet/model.py:147-153  */
#define SN_CELL_LSTM 1     /* gate blocks (i,f,g,o);  h = o*tanh(c)  nic/model.py:52,77         */

int32_t sn_version(void);
const char* sn_last_error(void);
/* device attributes the host side needs (SM count, opt-in shared memory, compute capability) */
int32_t sn_device_info(int32_t* sm_count, int32_t* smem_optin, int32_t* cc_major, int32_t* cc_minor);

/* ---- K1: embedding gather + dropout + feature row, packed time-major ------------------------
 * replaces self.B(captions); self.dropout(.); torch.cat((features.unsqueeze(1), .)) and the
 * per-step slicing embeddings[:b_sz, i, :]      stylenet/model.py:166-171,182; nic/model.py:85-89,101
 * row r -> sample row_b[r], step row_t[r].  has_feat: step 0 is the image feature row.
 * tok_override (optional, [N]): if >= 0 the row embeds that id instead (scheduled sampling feedback,
 * model.py:184) and is NOT dropped out.  X is [N, ldx] fp32; columns >= E are left untouched.
 * dropout: keep-prob 1-p, scale 1/(1-p), counter-based RNG (seed, row, col); p = 0 disables.
 * Xb (optional): the same rows as bf16 [N, ldxb], columns E..ldxb zero-filled (K padding of the tcgen05
 * operand); X may then be NULL.
 * seed_dev (optional, device): added to `seed` at run time -- lets a captured CUDA graph draw a fresh
 * mask on every replay (the caller bumps the device counter once per step). */
int32_t sn_gather_pack_fwd(const int64_t* captions, int64_t cap_ld, const float* table, int64_t E,
                           const float* features, int64_t feat_ld, int32_t has_feat,
                           const int32_t* row_b, const int32_t* row_t, const int32_t* tok_override,
                           int64_t N, float* X, int64_t ldx, float p_drop, uint64_t seed,
                           const uint64_t* seed_dev, void* Xb, int64_t ldxb, void* stream);
/* backward of the above: dtable[id] += dX*mask (atomic, duplicates accumulate like nn.Embedding's
 * dense gradient), dfeatures[b] = dX[row(b,0)] (may be NULL). */
int32_t sn_gather_pack_bwd(const int64_t* captions, int64_t cap_ld, float* dtable, int64_t E,
                           float* dfeatures, int64_t feat_ld, int32_t has_feat,
                           const int32_t* row_b, const int32_t* row_t, const int32_t* tok_override,
                           int64_t N, const float* dX, int64_t ldx, float p_drop, uint64_t seed,
                           const uint64_t* seed_dev, int64_t V, int32_t* ws_int, float* ws_part, void* stream);
/* Deterministic: the token rows are grouped by token (V = rows of dtable) and summed in row order, without float
   atomics.  Work space: ws_int 4*V + 1 + 3*N int32, ws_part (N/16 + 1)*E floats. */
/* sn_gather_pack_bwd in two parts.  The plan part groups the token rows by token: memset, count, scan, place and
   order into ws_int.  It reads only the captions, the packing plan and tok_override, so it can run as soon as those
   are final (in the forward, on a side stream).  The gradient part sums the groups from dX into dtable (zeroed by the
   caller) and writes dfeatures.  plan + grad is exactly sn_gather_pack_bwd.  wide != 0 sums each chunk of a group
   with one CTA of one thread per column (E <= 512; the same bits, a fraction of the latency). */
int32_t sn_embed_plan(const int64_t* captions, int64_t cap_ld, int32_t has_feat, const int32_t* row_b,
                      const int32_t* row_t, const int32_t* tok_override, int64_t N, int64_t V, int32_t* ws_int,
                      void* stream);
int32_t sn_embed_grad(float* dtable, int64_t E, float* dfeatures, int64_t feat_ld, int32_t has_feat,
                      const int32_t* row_b, const int32_t* row_t, const int32_t* tok_override, int64_t N,
                      const float* dX, int64_t ldx, float p_drop, uint64_t seed, const uint64_t* seed_dev, int64_t V,
                      const int32_t* ws_int, float* ws_part, int32_t wide, void* stream);

/* ---- K2: GEMM (all nn.Linear call sites: V_g/S_*_g/U_g model.py:119-150, C model.py:189-194,
 * encoder_att/decoder_att/f_beta/init_h/init_c model_att.py:59-61,192-193,283, LSTMCell's two
 * addmm nic/model.py:77) and every matmul autograd derives from them.
 * C = op(A) op(B) + bias[n] + beta*C, batched over `batch` groups with element strides.
 * A,B,C dtype: fp32 for SN_PREC_F32; see sn_gemm_tc for the tensor-core operand formats. */
int32_t sn_gemm(int32_t op, int64_t M, int64_t N, int64_t K, const float* A, int64_t lda,
                const float* B, int64_t ldb, float* C, int64_t ldc, const float* bias, float beta,
                int32_t batch, int64_t strideA, int64_t strideB, int64_t strideC, int64_t strideBias,
                void* stream);
/* The same GEMM on the tcgen05 tensor cores (SN_PREC_BF16): A, B are bf16 (row-major, leading dimensions
 * and group strides multiples of 8 elements, 16-byte aligned bases -- the TMA rules), accumulation is
 * fp32 in TMEM, the result is written as fp32 (C, may be NULL) and/or bf16 (Cb, may be NULL).
 * 1..4 groups.  TMA-fed (cp.async.bulk.tensor, 128B swizzle), K/M/N tails zero-filled / masked. */
int32_t sn_gemm_bf16(int32_t op, int64_t M, int64_t N, int64_t K, const void* A, int64_t lda,
                     const void* B, int64_t ldb, float* C, int64_t ldc, void* Cb, int64_t ldcb,
                     const float* bias, float beta, int32_t batch, int64_t strideA, int64_t strideB,
                     int64_t strideC, int64_t strideCb, int64_t strideBias, void* stream);
/* split-K variant of the single-CTA kernel (small M only; the CTA-pair kernel sn_gemm2_bf16 has its own
 * deterministic work-space split-K): the K loop is divided over `splits` CTAs per tile, partial tiles are
 * reduced with fp32 atomics into a zeroed C (fp32 output only, beta = 0; NOT bit-reproducible -- measured
 * slower than the work-space reduction for the weight-gradient GEMMs, profiles/README.md r1_d).  splits = 1: off. */
int32_t sn_gemm_bf16_splitk(int32_t op, int64_t M, int64_t N, int64_t K, const void* A, int64_t lda,
                            const void* B, int64_t ldb, float* C, int64_t ldc, void* Cb, int64_t ldcb,
                            const float* bias, float beta, int32_t batch, int64_t strideA,
                            int64_t strideB, int64_t strideC, int64_t strideCb, int64_t strideBias,
                            int32_t splits, void* stream);
/* K2b: the same GEMM as sn_gemm_bf16 on CTA PAIRS (tcgen05.mma.cta_group::2, 256x256 tiles, persistent tile loop,
 * double-buffered TMEM accumulator; sn_gemm2.cu).  Twice the arithmetic intensity per byte fetched from L2 --
 * the kernel for the time-batched projection / vocabulary / weight-gradient GEMMs (M >= 256).
 * splits > 1: split-K through the caller-provided work space `ws` (sn_gemm2_ws_bytes), reduced by a second
 * kernel (deterministic, no atomics); any epilogue (bias, beta, bf16 copy) is applied by the reduction.
 * max_pairs > 0 caps the grid at that many SM pairs (GEMMs on a side stream: leave SMs to the critical chain). */
int64_t sn_gemm2_ws_bytes(int64_t M, int64_t N, int32_t batch, int32_t splits);
int32_t sn_gemm2_bf16(int32_t op, int64_t M, int64_t N, int64_t K, const void* A, int64_t lda,
                      const void* B, int64_t ldb, float* C, int64_t ldc, void* Cb, int64_t ldcb,
                      const float* bias, float beta, int32_t batch, int64_t strideA, int64_t strideB,
                      int64_t strideC, int64_t strideCb, int64_t strideBias, int32_t splits, void* ws,
                      int64_t ws_bytes, int32_t max_pairs, void* stream);
/* fp32 [R,C] (row pitch lds) -> bf16 [R,Cp] (row pitch ldd), columns C..Cp zero-filled (weight shadows and
 * activation operands of sn_gemm_bf16; Cp pads K to the TMA 16-byte rule, e.g. E=300 -> 304) */
int32_t sn_cast_bf16(const float* src, int64_t R, int64_t C, int64_t lds, void* dst, int64_t Cp,
                     int64_t ldd, void* stream);
/* same, with the grid capped at max_blocks CTAs (0 = no cap): for casts issued on a side stream next to CTA-pair
 * GEMMs, which need whole SMs */
int32_t sn_cast_bf16_ex(const float* src, int64_t R, int64_t C, int64_t lds, void* dst, int64_t Cp,
                        int64_t ldd, int32_t max_blocks, void* stream);
/* column sums (bias gradients): out[n] = sum_m X[m,n] + beta*out[n] */
int32_t sn_colsum(const float* X, int64_t M, int64_t N, int64_t ldx, float* out, float beta,
                  void* stream);
int32_t sn_colsum_bf16(const void* X, int64_t M, int64_t N, int64_t ldx, float* out, float beta,
                       void* stream);
/* the same sums, bit for bit, with 16-byte loads (4 fp32 / 8 bf16 columns per thread) when wide != 0 and X and
   ldx are 16-byte aligned; otherwise the scalar kernel */
int32_t sn_colsum_ex(const float* X, int64_t M, int64_t N, int64_t ldx, float* out, float beta, int32_t wide,
                     void* stream);
int32_t sn_colsum_bf16_ex(const void* X, int64_t M, int64_t N, int64_t ldx, float* out, float beta, int32_t wide,
                          void* stream);

/* ---- K3: persistent recurrence (W_hh h + gates + cell), forward and reverse-time backward -----
 * replaces the hot loop stylenet/model.py:180-187 with forward_step's W_g(h_t)+sigmoid/tanh+cell
 * (model.py:147-153) resp. nn.LSTMCell (nic/model.py:77), for steps t0 <= t < t1.
 *   XP    [N,4H]  time-parallel input projection incl. its biases (U(S(V x)) + bU  /  x W_ih^T + b_ih)
 *   Whh   [4H,H]  W_i;W_f;W_o;W_c stacked (factored) / lstm.weight_hh
 *   bhh   [4H]    recurrent bias (bW_i..bW_c stacked / lstm.bias_hh), may be NULL
 *   h_init [B,H]  h before step t0 (NULL = zeros).  To continue a sequence at t0>0 pass the Hall rows
 *                 of step t0-1 (Hall + offsets[t0-1]*H)
 *   c_state [B,H] in/out: c before step t0 on entry (caller zero-fills / copies init_c), c after the
 *                 last step of each sample on return
 *   Hall  [N,H]   h_t per packed row (output; also the inter-SM exchange buffer)
 *   Call  [N,H]   c_t per packed row (output, needed by backward; may be NULL for inference)
 *   Hprev [N,H]   h_{t-1} per packed row (output, may be NULL) -- operand of dW_hh = dZ^T Hprev
 *   gates [N,4H]  post-activation i,f,o,c~ (output, may be NULL for inference)
 *   ws            >= sn_recur_ws_bytes() bytes of scratch; zeroed by the call itself */
int64_t sn_recur_ws_bytes(int64_t B, int64_t T);
int32_t sn_recur_fwd(int32_t cell, int64_t H, int64_t B, const int32_t* batch_sizes,
                     const int32_t* offsets, int32_t t0, int32_t t1, const float* XP,
                     const float* Whh, const float* h_init, const float* bhh, float* Hall,
                     float* Call, float* Hprev, float* gates, float* c_state, void* ws,
                     void* stream);
/* reverse-time backward for steps t1 > t >= t0.
 *   dHall [N,H]   dL/dh_t from everything downstream of the recurrence (vocab projection, attention)
 *   dZ    [N,4H]  output: dL/d(pre-activation) = dXP (feeds dW_hh, dU, dS, dV, dB GEMMs)
 *   dh_carry,dc_carry [B,H]  in/out: gradient flowing into h_{t1-1}.. from later steps (zeros at the
 *                 end of the sequence); on return hold dL/dh_{t0-1}, dL/dc_{t0-1} */
int32_t sn_recur_bwd(int32_t cell, int64_t H, int64_t B, const int32_t* batch_sizes,
                     const int32_t* offsets, int32_t t0, int32_t t1, const float* Whh,
                     const float* c_init, const float* Call, const float* gates, const float* dHall,
                     float* dZ, float* dh_carry, float* dc_carry, void* ws, void* stream);

/* bf16-mode variants of K3: W_hh (bf16 copy, [4H,H]) and the inter-SM exchange (h_t / dZ_t) are bf16, the
 * per-step contraction runs on the tensor cores with fp32 accumulation; state, gates and gradients fp32.
 *   Hb [N,H] bf16     h_t per packed row (output; exchange buffer and operand of the vocab projection)
 *   Hprevb [N,H] bf16 h_{t-1} per packed row (output, may be NULL)
 *   Hall [N,H] fp32   optional fp32 copy of h_t (may be NULL)
 *   dZb [N,4H] bf16   output: dXP in bf16 (exchange buffer and GEMM operand); dZ fp32 copy optional (NULL ok) */
int32_t sn_recur_fwd_bf16(int32_t cell, int64_t H, int64_t B, const int32_t* batch_sizes,
                          const int32_t* offsets, int32_t t0, int32_t t1, const float* XP,
                          const void* Whh_bf16, const float* bhh, const float* h_init, float* Hall,
                          void* Hb, void* Hprevb, float* Call, float* gates, float* c_state, void* ws,
                          void* stream);
int32_t sn_recur_bwd_bf16(int32_t cell, int64_t H, int64_t B, const int32_t* batch_sizes,
                          const int32_t* offsets, int32_t t0, int32_t t1, const void* Whh_bf16,
                          const float* c_init, const float* Call, const float* gates,
                          const float* dHall, float* dZ, void* dZb, float* dh_carry, float* dc_carry,
                          void* ws, void* stream);

/* K3, bf16 mode, CLUSTER form (sn_recur_cl.cu) -- same contract and arguments as sn_recur_{fwd,bwd}_bf16 (no work
 * space: nothing is exchanged through global memory).  Each slice of 16 samples runs inside one thread-block cluster
 * of H/32 CTAs for all steps: the bf16 W_hh slice of a CTA stays in registers, h_t (forward) / the fp32 dh partials
 * (backward) travel through distributed shared memory with st.async + mbarrier complete_tx.  Clusters are independent,
 * so there is no co-residency requirement (a plain launch cannot deadlock).  H in {128, 256, 512}.
 * replaces: stylenet/model.py:147-153,180-187 ; nic/model.py:77 (as above).
 * sn_recur_cl_max_clusters: how many such clusters the device can run at once (0 = form not available for this H). */
int32_t sn_recur_cl_max_clusters(int64_t H);
int32_t sn_recur_fwd_cl(int32_t cell, int64_t H, int64_t B, const int32_t* batch_sizes,
                        const int32_t* offsets, int32_t t0, int32_t t1, const float* XP,
                        const void* Whh_bf16, const float* bhh, const float* h_init, float* Hall,
                        void* Hb, void* Hprevb, float* Call, float* gates, float* c_state,
                        void* stream);
int32_t sn_recur_bwd_cl(int32_t cell, int64_t H, int64_t B, const int32_t* batch_sizes,
                        const int32_t* offsets, int32_t t0, int32_t t1, const void* Whh_bf16,
                        const float* c_init, const float* Call, const float* gates,
                        const float* dHall, float* dZ, void* dZb, float* dh_carry, float* dc_carry,
                        int32_t* start_flag, void* stream);
/* start_flag (may be NULL): 3 zero-initialised int32 words.  The backward kernel bumps word 1 once all its CTAs are
 * resident; sn_gate_wait (one spinning thread, queued on ANOTHER stream) returns when a bump it has not consumed yet
 * is there (or after timeout_us).  Work queued behind the gate -- the vocabulary weight gradient, bucket exchanges --
 * then starts on the SMs the clusters leave free instead of taking SMs the clusters still need. */
int32_t sn_gate_wait(int32_t* flag3, int64_t timeout_us, void* stream);

/* K3 in the LARGE-BATCH regime (B >= ~1000 samples per GPU): one tcgen05 CTA-pair GEMM per time step with the
 * cell fused into the epilogue, instead of the latency-optimised persistent kernel above.
 * replaces the same call sites: forward_step's W_g(h) + gate math  stylenet/model.py:119-153, nn.LSTMCell nic/model.py:77
 *   forward, step t:  Z = h_{t-1} Wp^T  (M = batch_sizes[t], N = 4H, K = H), epilogue adds XP_t + b_hh, applies the gate
 *     nonlinearities, updates c, writes h_t (fp32 + bf16), c_t and the activated gates.  Wp = W_hh with the rows of the
 *     four gate blocks interleaved 64 units at a time (sn_cast_bf16_gate_interleave): a 256-column accumulator tile
 *     then holds all four gates of 64 units and the epilogue warps of a lane quadrant exchange them through shared
 *     memory, so every global access of the cell update is a full 128-byte row segment.
 *   backward, step t: dh_rec = dZ_{t+1} W_hh (M = batch_sizes[t], N = H, K = 4H; rows of samples that ended at t read
 *     zeros), epilogue applies the cell backward and writes dZ_t (fp32 optional + bf16) and the carried dc.
 * bs_host / off_host: HOST copies of batch_sizes / offsets (the host issues one launch per step).  Whole sequences
 * only (t = 0..T-1, zero initial state).  zeros_bf16: >= max(B*H, 4H) zero bf16 elements.  H % 64 == 0. */
int32_t sn_cast_bf16_gate_interleave(const float* W, int64_t H, int64_t K, int64_t ldw, void* Wp,
                                     int64_t ldp, void* stream);
int32_t sn_recur_fwd_gemm(int32_t cell, int64_t H, int64_t B, const int32_t* bs_host,
                          const int32_t* off_host, int32_t T, const float* XP, const void* Wp_bf16,
                          const float* bhh, float* Hall, void* Hb, float* Call, float* gates,
                          const void* zeros_bf16, void* stream);
/* Hprevb[row(b,t)] = Hb[row(b,t-1)] (zeros at t = 0): the bf16 h_{t-1} operand of dW_hh = dZ^T Hprev */
int32_t sn_recur_hprev(const void* Hb, const int32_t* row_b, const int32_t* row_t,
                       const int32_t* offsets, int64_t N, int64_t H, void* Hprevb, void* stream);
int32_t sn_recur_bwd_gemm(int32_t cell, int64_t H, int64_t B, const int32_t* bs_host,
                          const int32_t* off_host, int32_t T, const void* Whh_bf16, const float* Call,
                          const float* gates, const float* dHall, float* dZ, void* dZb, float* dc_carry,
                          const void* zeros_bf16, void* stream);

/* ---- K5/K6: log-softmax + NLL (+ gradient) over logits, arg-max, top-5 ------------------------
 * replaces nn.CrossEntropyLoss (train_multitask.py:134,383), output.max(1) (model.py:190) and
 * utils.accuracy top-5 (utils.py:127-140).
 * row_loss[N] = lse - logit[target]; dlogits = (softmax - onehot) * grad_scale (may alias logits, may
 * be NULL); argmax[N] lowest index on ties (torch.max); top5hit[N] = 1 if fewer than 5 logits exceed
 * the target's.  targets may be NULL (then only argmax is produced).  dlogits_bf16 (optional, [N,lddb],
 * columns V..lddb zero): the gradient as the bf16 operand of the two vocab-projection backward GEMMs.
 * row_weight (optional, float [N], any sign): the gradient of row r is multiplied by row_weight[r] (the gradient of
 * sum_r w_r * row_loss_r * grad_scale); row_loss, argmax and top5hit do not depend on it.  NULL = weight 1, with the
 * arithmetic of a call without weights. */
int32_t sn_softmax_nll(const float* logits, int64_t N, int64_t V, int64_t ld, const int64_t* targets,
                       float* row_loss, float* dlogits, int64_t ldd, float grad_scale, const float* row_weight,
                       int64_t* argmax, int32_t* top5hit, void* dlogits_bf16, int64_t lddb, void* stream);
/* K5 fused with the vocabulary projection (bf16 mode): logits = Hb Wb^T + bias are produced tile by tile in
 * TMEM and consumed by the epilogue -- the [N,V] logits are NEVER written to HBM.
 * replaces self.C(hiddens) + nn.CrossEntropyLoss + output.max(1) + utils.accuracy
 *   stylenet/model.py:189-194, train_multitask.py:134,377-383, utils.py:127-140
 * sn_vocab_nll_fwd: per-row log-sum-exp `lse`, target logit `tlogit`, row_loss = lse - tlogit, argmax (lowest index
 *   on ties); `above` (optional) is zeroed for the ranking pass.  ws: sn_vocab_ws_bytes(N, V) bytes.
 * sn_vocab_nll_bwd: recomputes the logits tiles and writes dL = (softmax - onehot) * grad_scale as the bf16
 *   [N, lddl] operand of the two backward GEMMs (columns V..lddl zero; dL may be NULL = ranking only);
 *   above[row] += #{v : logit_v > logit_target}; top5hit[row] = above[row] < 5 (optional).
 *   row_weight (optional, float [N], any sign): dL of row r = (softmax - onehot) * grad_scale * row_weight[r], with
 *   log2(|w| * grad_scale) folded into the exponent offset and the sign applied after it (w = 0 writes zeros); NULL =
 *   the arithmetic of a call without weights.
 * Hb [N,ldh], Wb [V,ldw]: bf16, K = H padded per the TMA rules of sn_gemm_bf16. */
int64_t sn_vocab_ws_bytes(int64_t N, int64_t V);
int32_t sn_vocab_nll_fwd(int64_t N, int64_t V, int64_t H, const void* Hb, int64_t ldh, const void* Wb,
                         int64_t ldw, const float* bias, const int64_t* targets, void* ws, int64_t ws_bytes,
                         float* tlogit, float* lse, float* row_loss, int64_t* argmax, int32_t* above,
                         void* stream);
int32_t sn_vocab_nll_bwd(int64_t N, int64_t V, int64_t H, const void* Hb, int64_t ldh, const void* Wb,
                         int64_t ldw, const float* bias, const int64_t* targets, const float* tlogit,
                         const float* lse, float grad_scale, const float* row_weight, void* dL, int64_t lddl,
                         int32_t* above, int32_t* top5hit, void* stream);
/* loss = scale * sum(row_loss[0..N) * row_weight[0..N)) (+ loss if accumulate), deterministic order, double sum;
 * row_weight may be NULL (weight 1, the products are skipped) */
int32_t sn_reduce_sum(const float* x, int64_t N, float scale, const float* row_weight, float* out,
                      int32_t accumulate, void* stream);

/* ---- K7: fused clamp + Adam over flat parameter ranges ---------------------------------------
 * replaces utils.clip_gradient (utils.py:51-60) + torch.optim.Adam.step (train_multitask.py:388-389)
 * ranges: n_ranges x {offset,length} (int64 pairs, HOST memory) into the flat p/g/m/v arrays;
 * step_size[r] = lr/(1-beta1^t), bc2_sqrt[r] = sqrt(1-beta2^t) per range (HOST arrays).
 * torch op order: m.lerp_(g,1-b1); v.mul_(b2).addcmul_(g,g,1-b2); p.addcdiv_(m, sqrt(v)/bc2_sqrt+eps, -step_size) */
int32_t sn_adam_clamp(float* p, float* g, float* m, float* v, int32_t n_ranges,
                      const int64_t* ranges, const float* step_size, const float* bc2_sqrt,
                      float beta1, float beta2, float eps, float clip, void* stream);

/* Same kernel with the per-parameter step counters and the learning rate in DEVICE memory, so the whole
 * training step can be replayed from a CUDA graph: a prologue kernel increments steps_dev[step_idx[r]] and
 * derives lr/(1-beta1^t), sqrt(1-beta2^t) in double precision into coef_ws[2*step_idx[r]], [2*step_idx[r]+1]
 * (2 * (max step_idx + 1) floats: the slot belongs to the parameter, so calls that run concurrently on different
 * streams over disjoint parameters never share one). */
int32_t sn_adam_clamp_dev(float* p, float* g, float* m, float* v, int32_t n_ranges,
                          const int64_t* ranges, const int32_t* step_idx, int32_t* steps_dev,
                          const float* lr_dev, float* coef_ws, float beta1, float beta2, float eps,
                          float clip, void* stream);
/* same, with the grid capped at max_ctas CTAs of 256 threads (0 = the full 8 per SM): buckets updated on a side stream
   next to the critical chain leave it its SMs.  The grid size changes no element's result. */
int32_t sn_adam_clamp_dev_ex(float* p, float* g, float* m, float* v, int32_t n_ranges,
                             const int64_t* ranges, const int32_t* step_idx, int32_t* steps_dev,
                             const float* lr_dev, float* coef_ws, float beta1, float beta2, float eps,
                             float clip, int32_t max_ctas, void* stream);

/* ---- K9: data-parallel exchange fused with the optimizer, over NVLink peer memory (no NCCL) ------------
 * The reference has no distributed code; this replaces what `ncclAllReduce` + K7 would do.  Every rank (one
 * process per GPU) calls it with the SAME ranges after its backward: reduce-scatter of the gradient ranges by
 * peer loads (chunk c of 4096 elements is owned by rank c % world, summed in rank order 0..world-1), clamp +
 * Adam on the owned chunks (moments only for owned chunks), all-gather of the new parameters by peer stores.
 *   grad_ptrs/param_ptrs/pad_ptrs  HOST arrays of `world` DEVICE pointers: every rank's flat gradient arena,
 *                flat parameter arena and 32-int signal pad (zero-initialised once), mapped into this process
 *                (CUDA IPC) with peer access enabled (sn_enable_peer_access)
 * The kernel is also the cross-GPU barrier (arrive / done epoch flags in the pads, epoch kept in device memory),
 * so it is CUDA-graph replayable and must be called by all ranks the same number of times. */
int32_t sn_enable_peer_access(int32_t peer_device);
/* CUDA IPC plumbing for the above: export = (64-byte handle of the cudaMalloc allocation containing ptr, byte
 * offset of ptr in it); open maps that allocation into this process as a PEER mapping of the current device. */
int32_t sn_ipc_export(const void* ptr, uint8_t* handle64, int64_t* offset);
int32_t sn_ipc_open(const uint8_t* handle64, void** base_out);
int32_t sn_ipc_close(void* base);
int32_t sn_dp_adam_fused(int32_t world, int32_t rank, void* const* grad_ptrs, void* const* param_ptrs,
                         void* const* pad_ptrs, float* m, float* v, int32_t n_ranges,
                         const int64_t* ranges, const int32_t* step_idx, int32_t* steps_dev,
                         const float* lr_dev, float* coef_ws, float beta1, float beta2, float eps,
                         float clip, void* stream);
/* Push form of the same exchange, in two calls, so that the gradient transfer leaves the end of the step:
 *   sn_dp_push      (non-blocking) as soon as a bucket of gradient ranges is final, on the stream that produced it:
 *                   my gradients of the chunks I do not own go to their owners' receive buffers by posted NVLink
 *                   stores (fp32, or bf16 when elem_size == 2), then my ARRIVE flag is raised in every peer's pad of
 *                   this bucket.  Nothing waits: the transfer overlaps the rest of the backward.
 *   sn_dp_adam_recv for a set of pushed buckets (1..4): waits (local polls) until every peer's pushes of those buckets
 *                   have landed, reduces own fp32 gradient + the received ones in rank order, clamp + Adam on the owned
 *                   chunks, parameter all-gather by peer stores, exit barrier (DONE flags in the pads of wait bucket 0).
 *   recv_ptrs    every rank's receive buffer: `world` slots of sn_dp_slot_elems(arena_elems, world) elements; slot q of
 *                rank o holds rank q's gradients of o's chunks, chunk `aid` at element (aid / world) * 4096
 *   pad_ptrs     every rank's pad of the bucket (push) / of wait bucket 0 (recv); wait_pads: MY pads of the consumed
 *                buckets, wait_pads[0] == pad_ptrs[rank]
 *   max_ctas     0 = the whole GPU (exchange at the end of the step); > 0 caps the grid (1024-thread CTAs for the push,
 *                512-thread CTAs for the receive side) for an exchange that runs UNDER the backward and must leave the
 *                GEMMs their SMs
 * With elem_size 4 the sum is bit-identical to sn_dp_adam_fused's (same operands, same order). */
int64_t sn_dp_slot_elems(int64_t arena_elems, int32_t world);
int32_t sn_dp_push(int32_t world, int32_t rank, const float* grad, void* const* recv_ptrs, int64_t slot_elems,
                   int32_t elem_size, void* const* pad_ptrs, int32_t n_ranges, const int64_t* ranges,
                   int32_t max_ctas, void* stream);
int32_t sn_dp_adam_recv(int32_t world, int32_t rank, float* grad, void* const* param_ptrs, void* recv,
                        int64_t slot_elems, int32_t elem_size, void* const* pad_ptrs, void* const* wait_pads,
                        int32_t n_wait, float* m, float* v, int32_t n_ranges, const int64_t* ranges,
                        const int32_t* step_idx, int32_t* steps_dev, const float* lr_dev, float* coef_ws,
                        float beta1, float beta2, float eps, float clip, int32_t max_ctas, void* stream);

/* ---- K4: soft attention step (scores -> softmax over pixels -> context -> f_beta gate) ----------
 * replaces Attention.forward after the hoisted encoder_att GEMM (model_att.py:61-70) and the gate
 * multiply (model_att.py:283-284) for one time step over nb samples.
 *   att1 [B,P,A] (= encoder_att(features), time-invariant), att2 [nb,A] (= decoder_att(h)),
 *   feat [B,P,D], wfull [A], bfull scalar, gate_pre [nb,D] (= f_beta(h), pre-sigmoid)
 *   alpha [nb,P] out, ctx [nb, ldc] out = sigmoid(gate_pre) * sum_p alpha_p feat_p */
int32_t sn_att_step_fwd(const float* att1, const float* att2, const float* feat, const float* wfull,
                        float bfull, const float* gate_pre, int64_t nb, int64_t P, int64_t A,
                        int64_t D, float* alpha, int64_t ld_alpha, float* ctx, int64_t ldc,
                        void* stream);
/* backward of one attention step.  Inputs as forward plus dctx [nb, ldc] and dalpha_extra [nb,P]
 * (gradient of the doubly-stochastic regulariser, may be NULL).  Outputs: datt2 [nb,A], dgate_pre
 * [nb,D], datt1 [B,P,A] ACCUMULATED (+=), dwfull [A] ACCUMULATED via atomics, dfeat (may be NULL)
 * ACCUMULATED. */
int32_t sn_att_step_bwd(const float* att1, const float* att2, const float* feat, const float* wfull,
                        float bfull, const float* gate_pre, const float* alpha, int64_t ld_alpha,
                        const float* dctx, int64_t ldc, const float* dalpha_extra, int64_t ld_da,
                        int64_t nb, int64_t P, int64_t A, int64_t D, float* datt2, float* dgate_pre,
                        float* datt1, float* dwfull, float* dfeat, void* stream);
/* mean over pixels: out[b,d] = mean_p feat[b,p,d]   (model_att.py:191) */
int32_t sn_mean_pixels(const float* feat, int64_t B, int64_t P, int64_t D, float* out, void* stream);

/* ---- K8: beam / greedy decode bookkeeping -----------------------------------------------------
 * replaces log_softmax + running-score add + topk + index arithmetic + the host-side completion loop
 * of sample() (stylenet/model.py:232-285; model_att.py:364-417; nic/model.py:145-198) for a BATCH of
 * images, one step, with no host synchronisation.  Rows of image i are [i*kmax, (i+1)*kmax); the first
 * k_live[i] rows are its live beams in top-k order.  L = max_len + 2 ints per sequence.
 *   logits [n_img*kmax, ld]   this step's C(h) for every row (dead rows ignored)
 *   k_live [n_img]            in/out live beam count (k shrinks as beams finish; 0 = image finished)
 *   run_score/prev_word/src_row [n_img*kmax]   in/out running log-prob, the word to feed next, and the
 *                             row whose (h,c) the beam continues from (caller gathers state with it)
 *   cur_buf [n_img], seqs [2][n_img*kmax][L]    double-buffered partial sequences
 *   done_seq/done_len/done_score/n_done         finished beams in completion order
 *   out_seq [n_img][L], out_len [n_img]         final result when the image finishes: first arg-max of
 *                             the un-normalised scores of finished beams, or [end] if none finished
 *   n_unfinished [1]          decremented once per image when it finishes (poll to stop early)
 * step counts from 1; an image finishes when k reaches 0 or after step > max_len (model.py:273,283).
 * step_dev (optional, device int): the step number read at run time instead of `step`, so that one captured
 * decode step can be replayed from a CUDA graph (the caller increments it on the device). */
int32_t sn_beam_step(const float* logits, int64_t ld, int64_t V, int32_t n_img, int32_t kmax,
                     int32_t step, int32_t max_len, int32_t end_token, int32_t* k_live,
                     float* run_score, int32_t* prev_word, int32_t* src_row, int32_t* cur_buf,
                     int32_t* seqs, int32_t* done_seq, int32_t* done_len, float* done_score,
                     int32_t* n_done, int32_t* out_seq, int32_t* out_len, int32_t* n_unfinished,
                     const int32_t* step_dev, void* stream);

/* K4 with a bf16 feature map (bf16 mode): same contract as sn_att_step_fwd / _bwd, `feat_bf16` [B,P,D] bf16 (half the
 * bytes of the largest tensor of the step, read with 16-byte loads); att1 / att2 / the relu pre-activation stay fp32.
 * No d feat output.  Needs D == 2048, A % 4 == 0, 16-byte aligned rows; returns -2 when not applicable. */
int32_t sn_att_step_fwd_b16(const float* att1, const float* att2, const void* feat_bf16, const float* wfull,
                            float bfull, const float* gate_pre, int64_t nb, int64_t P, int64_t A, int64_t D,
                            float* alpha, int64_t ld_alpha, float* ctx, int64_t ldc, void* stream);
int32_t sn_att_step_bwd_b16(const float* att1, const float* att2, const void* feat_bf16, const float* wfull,
                            const float* gate_pre, const float* alpha, int64_t ld_alpha, const float* dctx,
                            int64_t ldc, const float* dalpha_extra, int64_t ld_da, int64_t nb, int64_t P,
                            int64_t A, int64_t D, float* datt2, float* dgate_pre, float* datt1,
                            float* dwfull, void* stream);

/* sn_beam_step for FEW images: the same step spread over nch x more CTAs (per-chunk log-sum-exp partials, per-chunk
 * top-k of the final scores, per-image merge + bookkeeping).  Same arguments as sn_beam_step plus the chunk count
 * (1..32) and a work space of sn_beam_split_ws_floats() floats.  Same selection rule (score descending, ties -> lower
 * flat index); the log-sum-exp is combined from chunk partials, so scores may differ from sn_beam_step in the last bit.
 * advance_step != 0 (needs step_dev): the last block adds 1 to *step_dev; the work space must be zero-filled once. */
int64_t sn_beam_split_ws_floats(int32_t n_img, int32_t kmax, int32_t nch);
int32_t sn_beam_step_split(const float* logits, int64_t ld, int64_t V, int32_t n_img, int32_t kmax,
                           int32_t step, int32_t max_len, int32_t end_token, int32_t* k_live,
                           float* run_score, int32_t* prev_word, int32_t* src_row, int32_t* cur_buf,
                           int32_t* seqs, int32_t* done_seq, int32_t* done_len, float* done_score,
                           int32_t* n_done, int32_t* out_seq, int32_t* out_len, int32_t* n_unfinished,
                           const int32_t* step_dev, int32_t nch, float* ws, int32_t advance_step,
                           void* stream);

/* ---- SN_PREC_BF16X6: limb expansion of fp32 GEMM operands (see sn_split.cu) ------------------------------------
 * x = x0 + x1 + x2 (bf16 limbs); left operands get the slots [x1 x0 x2 x0 x1 x0], right operands [x1 x2 x0 x1 x0 x0]
 * along the contraction dimension, so ONE bf16 GEMM with K' = 6*Kp evaluates a1b1+a0b2+a2b0+a0b1+a1b0+a0b0 in fp32
 * (smallest products first: the tensor core's accumulator alignment truncates relative to the running sum).
 *   _cols: K runs along the columns.  src [R, G*K] (pitch ld) -> dst bf16 [R, G*6*Kp] (Kp = K padded to 8, zeros)
 *   _rows: K runs along the rows.     src [G*K, C] (pitch ld) -> dst bf16 [G*6*Kp, Cp]  (Cp = C padded to 8, zeros)
 * pattern: 0 = left operand, 1 = right operand. */
int32_t sn_split_limbs_cols(const float* src, int64_t R, int64_t G, int64_t K, int64_t ld, void* dst,
                            int64_t Kp, int32_t pattern, void* stream);
int32_t sn_split_limbs_rows(const float* src, int64_t G, int64_t K, int64_t C, int64_t ld, void* dst,
                            int64_t Kp, int64_t Cp, int32_t pattern, void* stream);

/* ---- decode steps on FEW rows (single-image beam search, forward_step): matrix-vector kernels -----------------
 * replaces forward_step (stylenet/model.py:115-155, nn.LSTMCell nic/model.py:77) and the per-step C(h)
 * (model.py:234) when rows <= sn_skinny_max_rows(): one pass over the fp32 weights, rows held in shared memory.
 * sn_skinny_linear: out[r,n] = bias[n] + W[n,:K] . X[r, xoff(n) : xoff(n)+K], xoff(n) = (n / group_n) * group_x
 *   (group_n = 0: no groups; the four S_g / U_g blocks are groups of F resp. H features reading column block g).
 *   x_rows (may be NULL): row r of the input is X[x_rows[r]] -- the embedding lookup of the previous words
 *   (stylenet/model.py:231) folded into the first stage.
 * sn_decode_cell: z_g = Wx[g*H+u,:Kx] . x_g[r] + bx + Wh[g*H+u,:] . h_prev[src_row[r]] + bh, gates, c', h' for
 *   every unit u and row r; x_g = X[r, g*group_x : +Kx] (group_x = 0: the same x for all gates, LSTMCell).
 *   src_row (may be NULL) re-orders the incoming state per row (beam bookkeeping, model.py:275-279): h_out / c_out
 *   must not alias h_prev / c_prev.  x_rows (may be NULL): row r of the input is X[x_rows[r]] -- with the factored
 *   chain collapsed once per decode call (Wx = U_g S_g V_g, bx = U_g(S_g bV_g + bS_g) + bU_g) the embedding lookup,
 *   the three projection stages and the cell are this one kernel.
 *   sn_skinny_linear also takes more than sn_skinny_max_rows() rows (up to 256): balanced chunks of <= 16 rows along
 *   grid.y, each chunk computed exactly as a call on those rows alone.
 * sn_decode_cell_groups: sn_decode_cell for G <= 4 row groups in ONE launch -- the per-style sample() calls of one
 *   image (app/backend/model.py's four get_sample calls per upload; forward_step, stylenet/model.py:115-155, with the
 *   style's S in the chain) as one decode step.  Group g owns rows [row_off[g], row_off[g+1]) (row_off: device int32
 *   [G+1], non-decreasing) and reads Wx + g*sWx, bx + g*sbx (the collapsed chain of its style); W_hh, b_hh, src_row,
 *   x_rows and the state are shared over all rows, as in sn_decode_cell.  rows_max >= the largest group (host-known,
 *   sizes the row chunks).  Each row's arithmetic is that of sn_decode_cell: a step of the mixed rows equals the
 *   single-style step of the same rows bit for bit. */
int32_t sn_skinny_max_rows(void);
int32_t sn_skinny_linear(const float* W, int64_t ldw, int64_t N, int64_t K, const float* X, int64_t ldx,
                         int64_t R, int64_t group_n, int64_t group_x, const float* bias, float* out,
                         int64_t ldo, const int32_t* x_rows, void* stream);
int32_t sn_decode_cell(int32_t cell, int64_t H, int64_t R, const float* Wx, int64_t ldwx, int64_t Kx,
                       const float* X, int64_t ldx, int64_t group_x, const float* bx, const float* Wh,
                       const float* bh, const float* h_prev, const float* c_prev, const int32_t* src_row,
                       const int32_t* x_rows, float* h_out, float* c_out, void* stream);
int32_t sn_decode_cell_groups(int32_t cell, int64_t H, int64_t G, const int32_t* row_off, int64_t rows_max,
                              const float* Wx, int64_t ldwx, int64_t sWx, int64_t Kx, const float* X, int64_t ldx,
                              int64_t group_x, const float* bx, int64_t sbx, const float* Wh, const float* bh,
                              const float* h_prev, const float* c_prev, const int32_t* src_row, const int32_t* x_rows,
                              float* h_out, float* c_out, void* stream);

/* ---- encoder tail -> decoder hand-off (SURVEY.md section 8 f1) ---------------------------------------------------
 * sn_pool_nhwc_fwd: AdaptiveAvgPool2d((S,S)) + permute(0,2,3,1) of the trunk output (stylenet/model_att.py:24-28),
 *   one pass: x [B,D,h,w] (NCHW) -> out [B,S,S,D] contiguous fp32, optional bf16 copy (GEMM operand) and optional
 *   mean over the S*S pixels [B,D] (what init_hidden_state needs, model_att.py:185-194).  h*w <= 1024.
 * sn_pool_nhwc_bwd: its backward (dx [B,D,h,w]); only needed when the trunk is fine-tuned.
 * sn_bn1d_fwd / _bwd: BatchNorm1d(E, momentum) behind Linear(2048,E) (stylenet/model.py:19-26): batch statistics +
 *   running-statistics update when training != 0, running statistics otherwise.  save_mean / save_invstd [E] feed
 *   the backward (pass the running mean and rsqrt(running_var + eps) in eval mode). */
int32_t sn_pool_nhwc_fwd(const float* x, int64_t B, int64_t D, int64_t h, int64_t w, int64_t S, float* out,
                         void* out_bf16, float* mean, void* stream);
int32_t sn_pool_nhwc_bwd(const float* dout, int64_t B, int64_t D, int64_t h, int64_t w, int64_t S, float* dx,
                         void* stream);
int32_t sn_bn1d_fwd(const float* x, int64_t B, int64_t E, const float* gamma, const float* beta,
                    float* running_mean, float* running_var, float momentum, float eps, int32_t training,
                    float* y, float* save_mean, float* save_invstd, void* stream);
int32_t sn_bn1d_bwd(const float* x, const float* dy, int64_t B, int64_t E, const float* gamma,
                    const float* save_mean, const float* save_invstd, int32_t training, float* dx,
                    float* dgamma, float* dbeta, void* stream);

/* ---- K10: corpus-BLEU n-gram statistics (sn_bleu.cu) -------------------------------------------------------------
 * replaces the per-hypothesis loop of nltk's corpus_bleu -- modified_precision and closest_ref_length
 * (nltk/translate/bleu_score.py) -- called by the reference at the end of every validation epoch
 * (stylenet/train_multitask.py:341, evaluator.py:103).
 * Inputs in CSR form (device memory): hypothesis i is hyp_tok[hyp_off[i] .. hyp_off[i+1]) and owns the references
 * ref_group[i] .. ref_group[i+1]-1; reference r is ref_tok[ref_off[r] .. ref_off[r+1]).  The references of one
 * hypothesis are contiguous.  max_sentence_len (longest hypothesis or reference, <= SN_BLEU_MAX_LEN) and
 * max_group_tokens (largest hypothesis length + total length of its references, sizes shared memory) are computed
 * by the caller while packing; either limit exceeded -> rc < 0 before any launch.
 * Output stats [n_hyp, 10] int32, per hypothesis:
 *   0..3  clipped n-gram matches, n = 1..4: sum over distinct hypothesis n-grams g of
 *         min(count_hyp(g), max over references of count_ref(g))         (modified_precision numerator)
 *   4..7  max(1, len_hyp - n + 1)                                         (modified_precision denominator)
 *   8     len_hyp
 *   9     closest reference length: minimises (|len_ref - len_hyp|, len_ref), ties -> the shorter reference
 *         (closest_ref_length); 0 for a hypothesis without references
 * Integer arithmetic, no atomics: exact and run-to-run identical.  Corpus totals are column sums.  A hypothesis
 * whose sizes exceed the declared maxima gets -1 in every column. */
#define SN_BLEU_MAX_LEN 256
int32_t sn_bleu_counts(const int32_t* hyp_tok, const int64_t* hyp_off, int64_t n_hyp,
                       const int32_t* ref_tok, const int64_t* ref_off, const int64_t* ref_group,
                       int32_t max_sentence_len, int64_t max_group_tokens, int32_t* stats, void* stream);

/* ---- K11: CIDEr-D (sn_cider.cu) -----------------------------------------------------------------------------------
 * replaces coco-caption's CiderScorer (pycocoevalcap/cider/cider_scorer.py, Cider(n, sigma).compute_score) on integer
 * token ids, document frequencies from the evaluated corpus.  Same CSR inputs as K10 (image i = hypothesis i and its
 * references; sn_cider_df reads only the references), the same limits (max_sentence_len <= SN_BLEU_MAX_LEN, an
 * image's tokens must fit in opt-in shared memory; either exceeded -> rc < 0 before any launch) and 1 <= n <= 4.
 * Token ids must be non-negative: -1 pads the keys of the document-frequency table.
 *
 * sn_cider_df -- compute_doc_freq: counts[s] = number of images whose references contain the n-gram keys[s, :],
 *   orders 1..n.  The table is caller memory: keys int32 [capacity, 4] (16-byte aligned; an n-gram of order k holds
 *   its k ids followed by -1s, an empty slot is all -1), counts int32 [capacity], capacity a power of two (at least
 *   2 x the number of reference n-grams keeps probe chains short).  The call clears the table and *err, then inserts
 *   each n-gram of an image's references at its first occurrence across them (one int32 atomic add per image): the
 *   counts are exact and independent of launch order.  Keys are compared in full; the hash only picks the first slot.
 *   *err (device int32, read it after the stream): |1 the table is full (counts are then incomplete), |2 a negative
 *   token id, |4 an image's sizes exceed the declared maxima.
 * sn_cider_scores -- compute_cider: per image, in float64, with ref_len = log(n_img) and
 *   idf(g) = ref_len - log(max(1, counts[g])) (an n-gram absent from the table has idf ref_len):
 *   counts2vec  vec[g] = tf(g) * idf(g) over the distinct n-grams of a sentence, norm[k] = sqrt(sum vec^2 of order k),
 *               length = number of bigrams (0 when n = 1: the scorer measures length on order index 1);
 *   sim         val[k] = sum over hypothesis n-grams g of min(vec_h[g], vec_r[g]) * vec_r[g], divided by
 *               norm_h[k] * norm_r[k] when both are non-zero, times e^(-(len_h - len_r)^2 / (2 sigma^2));
 *   per_order[i, k] = sum of val[k] over the references of image i (k < n; 0 for k >= n; may be NULL),
 *   scores[i]       = mean over the n orders of per_order[i, :] / (number of references) * 10.
 *   Fixed summation order, no float atomics: run-to-run bitwise identical.  An image whose sizes exceed the declared
 *   maxima gets NaN.  The corpus score is the mean of scores[]. */
int32_t sn_cider_df(const int32_t* ref_tok, const int64_t* ref_off, const int64_t* ref_group, int64_t n_img,
                    int32_t n, int32_t max_sentence_len, int64_t max_group_tokens, int32_t* keys, int32_t* counts,
                    int64_t capacity, int32_t* err, void* stream);
int32_t sn_cider_scores(const int32_t* hyp_tok, const int64_t* hyp_off, int64_t n_img, const int32_t* ref_tok,
                        const int64_t* ref_off, const int64_t* ref_group, int32_t n, double sigma,
                        int32_t max_sentence_len, int64_t max_group_tokens, const int32_t* keys,
                        const int32_t* counts, int64_t capacity, double* scores, double* per_order, void* stream);
/* sn_cider_scores_rows -- sn_cider_scores for R sampled captions against the references of the corpus the table was
 *   built from: row r's hypothesis is seqs[r, 1 .. lengths[r]) (int64 [R, ld]; column 0 holds <start>) without a final
 *   end_token, scored against the references of image img[r] (int64 [R], 0 <= img[r] < n_corpus), with
 *   ref_len = log(n_corpus) -- the corpus' image count, not R.  ref_off / ref_group are the corpus' CSR (ref_group has
 *   n_corpus + 1 entries).  max_sentence_len >= ld - 1 and the longest reference; max_group_tokens >= ld - 1 plus the
 *   largest reference token count of an image used.  The body is sn_cider_scores': with img[r] = r, n_corpus = R and
 *   the same hypotheses, the scores are bitwise equal. */
int32_t sn_cider_scores_rows(const int64_t* seqs, int64_t ld, const int64_t* lengths, int64_t R, int32_t end_token,
                             const int64_t* img, int64_t n_corpus, const int32_t* ref_tok, const int64_t* ref_off,
                             const int64_t* ref_group, int32_t n, double sigma, int32_t max_sentence_len,
                             int64_t max_group_tokens, const int32_t* keys, const int32_t* counts, int64_t capacity,
                             double* scores, void* stream);

/* ---- K13: ROUGE-L (sn_rouge.cu) -----------------------------------------------------------------------------------
 * replaces coco-caption's Rouge scorer (pycocoevalcap/rouge/rouge.py, Rouge().compute_score: my_lcs + calc_score) on
 * integer token ids.  Same CSR inputs as K10; max_sentence_len (longest hypothesis or reference) <= SN_BLEU_MAX_LEN,
 * else rc < 0 before any launch.  There is no per-image token limit: nothing is staged in shared memory.  Any int32 id
 * is valid (ids are only compared for equality).
 * sn_rouge_l -- per image i, with lcs_r = the longest common subsequence of hypothesis i and its reference r (exact,
 *   bit-parallel), len = the token count, an empty sentence counting as one token that only another empty sentence
 *   shares ("".split(" ") == [""]):
 *     p = max_r lcs_r / len_hyp,  r = max_r (lcs_r / len_ref_r),
 *     scores[i] = ((1 + beta2) * p * r) / (r + beta2 * p) if p != 0 and r != 0, else 0,
 *   every operation one correctly rounded float64 operation in that order (no FMA contraction), so the scores equal
 *   the scorer's bit for bit when beta2 is its beta**2 (1.2 ** 2).  No atomics: run-to-run identical.  An image whose
 *   sizes exceed the declared maximum, or without references, gets NaN.  The corpus score is the mean of scores[].
 * sn_rouge_l_rows -- the same body for R sampled captions against the references of a corpus (sn_cider_scores_rows'
 *   layout): row r's hypothesis is seqs[r, 1 .. lengths[r]) (int64 [R, ld]; column 0 holds <start>) without a final
 *   end_token, scored against the references of image img[r] (int64 [R], 0 <= img[r] < n_corpus; NaN otherwise).
 *   ld - 1 <= max_sentence_len.  With img[r] = r and the same hypotheses, the scores equal sn_rouge_l's bit for bit. */
int32_t sn_rouge_l(const int32_t* hyp_tok, const int64_t* hyp_off, int64_t n_img, const int32_t* ref_tok,
                   const int64_t* ref_off, const int64_t* ref_group, int32_t max_sentence_len, double beta2,
                   double* scores, void* stream);
int32_t sn_rouge_l_rows(const int64_t* seqs, int64_t ld, const int64_t* lengths, int64_t R, int32_t end_token,
                        const int64_t* img, int64_t n_corpus, const int32_t* ref_tok, const int64_t* ref_off,
                        const int64_t* ref_group, int32_t max_sentence_len, double beta2, double* scores,
                        void* stream);

/* ---- K12: sampling decode step (sn_sample.cu) ---------------------------------------------------------------------
 * One draw per live row r of logits [R, ld] (the step's vocabulary projection, V columns), for self-critical training:
 *   greedy = 0: token = argmax_v (logit_v / temperature + g_v), Gumbel-max;
 *   greedy = 1: token = argmax_v logit_v;
 *   ties go to the lowest index.  The noise is computed in double:
 *     seed_t = seed * 0x9E3779B97F4A7C15 + step        (uint64, wrapping)
 *     u      = ((hash_u32(seed_t, r, v) >> 8) + 0.5) / 2^24     (hash_u32: the dropout hash of sn_common.cuh)
 *     g_v    = -log(-log(u))
 *   seed (uint64) and step (int32, the 1-based draw index) are read from device memory (*seed_dev, *step_dev), so a
 *   captured CUDA graph of the step draws fresh noise when the counter moves.  The caller advances *step_dev.
 * Row bookkeeping (rows with done[r] != 0 are skipped; a row's draws go to column `step` of its sequence):
 *   seqs[r, step] = token (int64 [R, max_len + 2], column 0 = <start>), prev_word[r] = token (int32, the next input),
 *   logprob[r, step - 1] = logit_token - logsumexp(logits) (temperature 1; float [R, max_len + 1]);
 *   when token == end_token or step == max_len + 1: done[r] = 1, lengths[r] = step + 1, atomicSub(n_unfinished, 1). */
int32_t sn_sample_step(const float* logits, int64_t ld, int64_t V, int32_t R, int32_t max_len, int32_t end_token,
                       double temperature, int32_t greedy, const uint64_t* seed_dev, const int32_t* step_dev,
                       int32_t* prev_word, int64_t* seqs, int64_t* lengths, float* logprob, int32_t* done,
                       int32_t* n_unfinished, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SN100_H_ */
