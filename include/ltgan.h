/*
 * ltgan.h -- C ABI of the B200-native Long-Tail-GAN hot path (libltgan.so).
 *
 * The reference (ash-shar/Long-Tail-GAN) has no native boundary: its hot path is a TensorFlow-1 graph driven by
 * `sess.run` from Codes/train.py and Codes/test.py. Each entry point below replaces the TF ops (and the host NumPy
 * loops) cited next to it; the Python host layer in long-tail-gan_b200/ binds them with ctypes and keeps the
 * reference's plugin surface (generator.py / discriminator.py / sample.py / eval_functions.py signatures).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in _host; the caller owns all buffers, kernels allocate nothing
 *   - `stream` is a cudaStream_t passed as void*; all ops are asynchronous and stream-ordered (CUDA-graph capturable)
 *   - return 0 on success, negative on error (LTG_ERR_*); ltg_last_error() describes the last failure of this thread
 *   - bf16 tensors are row-major with the stated pitch ("ld", in elements); a pitch must be a multiple of 8 elements
 *   - H = 600 (hidden), L = 200 (latent) are the VAE-CF sizes hard-coded by generator.py:13
 *   - randomness is stateless Philox4x32-10 keyed by (seed, stream id, step, element index); `*_step_dev` arguments
 *     are optional device words added to the scalar step so that a captured CUDA graph can be replayed
 */
#ifndef LTGAN_H_
#define LTGAN_H_
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LTG_H 600
#define LTG_L 200

/* slots of the per-step fp32 scalar buffer (`scal`, at least LTG_NSCAL floats, zeroed by the caller per step) */
enum {
  LTG_S_KL_SUM = 0,   /* sum_u KL_u                      MultiVAE.py:161-162 (before the batch mean) */
  LTG_S_NLL_SUM = 1,  /* sum_u -sum_i x_ui log_softmax   MultiVAE.py:110-112 (before the batch mean) */
  LTG_S_SUM_P = 2,    /* sum over sampled (u,i) of softmax prob   train.py:145-149 */
  LTG_S_SUM_Y = 3,    /* sum over valid generated pairs of y      train.py:155 */
  LTG_S_CNT = 4,      /* number of valid generated pairs (sampled_cnt)  train.py:251,316; counted by ltg_disc_head */
  LTG_S_D_LOSS = 5,   /* d_loss  train.py:142 */
  LTG_S_LR_T = 8,     /* Adam: lr*sqrt(1-b2^t)/(1-b1^t), written by ltg_step_advance */
  LTG_S_ANNEAL = 9,   /* KL anneal weight of this G step, written by ltg_step_advance */
  LTG_NSCAL = 16
};

/* ---- runtime -------------------------------------------------------------------------------------------------- */
const char* ltg_last_error(void);
int ltg_version(void);
/* One-time per process and device: resolves cuTensorMapEncodeTiled, opts kernels into large shared memory. */
int ltg_init(void);

/* Persistent step state (device): words[0] = rng step, words[1] = Adam step t (shared by D and G updates, F6),
 * words[2] = G-update count (KL anneal, train.py:319-324). ltg_step_advance bumps the counters on the device and
 * writes LTG_S_LR_T / LTG_S_ANNEAL into `scal` after zeroing its accumulator slots [0, 8), so a captured graph needs no host values.
 *   kind: 0 = phase-A (rng only), 1 = D update (rng + Adam t), 2 = G update (rng + Adam t + anneal count)
 * zero_buf / zero_words: optional 4-byte-aligned buffer cleared by the same launch (the phase's atomically accumulated
 * gradients or counters), so no separate memset sits at the head of the phase.
 * step_snapshot: optional word that receives the new rng step; the phase's kernels take it as their `step_dev`, so phases whose
 * kernels overlap in time (the G forward beside the D update of the same batch, engine.run_step) each see their own step. */
int ltg_step_advance(uint32_t* words, float* scal, int kind, float lr, float beta1, float beta2,
                     float anneal_cap, float total_anneal_steps, void* zero_buf, int64_t zero_words, uint32_t* step_snapshot,
                     void* stream);
/* The advances of one whole A -> D -> G step in one launch: identical in effect to ltg_step_advance with kind 0, 1, 2 in this order
 * on three DISTINCT scalar rows (phase A's row is scratch: train.py:200 fetches no loss), each with its own cleared buffer and rng-step
 * snapshot. Used by the per-batch step graph (train.py:192-329 for one batch), where it takes two launches off the critical chain.  */
int ltg_step_advance3(uint32_t* words, float* scal_a, float* scal_d, float* scal_g, float lr, float beta1, float beta2,
                      float anneal_cap, float total_anneal_steps, void* zero_a, int64_t zero_a_words, void* zero_d,
                      int64_t zero_d_words, void* zero_g, int64_t zero_g_words, uint32_t* snap_a, uint32_t* snap_d,
                      uint32_t* snap_g, void* stream);

/* ---- generic bf16 tensor-core GEMM (tcgen05/TMA/TMEM) ------------------------------------------------------------
 * D[M,N] = alpha * A * B^T with A given as [M,K] (a_mn=0, pitch lda) or stored transposed [K,M] (a_mn=1), B likewise
 * ([N,K] or [K,N]); epilogue: +bias[N], act (0 none / 1 tanh), dropout(keep) from a counter hash of (row*rng_ld+col)/2, outputs fp32
 * and/or bf16; split-K either accumulates with `atomic` into a zeroed fp32 buffer or (split_stride > 0) stores the partial of
 * split s at out_f32 + s*split_stride for the consumer to sum; column `aux_col` is diverted to aux_out[row].
 * dact_src (bf16 [M, dact_ld], may be NULL): multiply the result by d/da dropout(tanh(a)) recovered from the stored
 * post-dropout activation (backward of discriminator.py:25,30,44 fused into the dgrad GEMM).
 * bn in {64,128,192,256}. Building block of every dense layer below (tf.matmul sites: MultiVAE.py:152,169;
 * discriminator.py:25-55) and their autodiff transposes (train.py:163-164).                                        */
int ltg_gemm_bf16(const void* A, int lda, int a_mn, const void* B, int ldb, int b_mn, int M, int N, int K, int splits, int bn,
                  float* out_f32, int ld_f32, void* out_bf16, int ld_bf16, const float* bias, int act, float alpha, int atomic,
                  float keep, uint64_t seed, uint32_t rng_stream, uint32_t rng_step, const uint32_t* rng_step_dev, int rng_ld,
                  int aux_col, float* aux_out, const void* dact_src, int dact_ld, float dact_keep, int64_t split_stride, void* stream);

/* ---- a3: encoder (MultiVAE.py:148-155): l2_normalize + dropout + x*W_q0 + b + tanh, as a CSR gather-sum -----------
 * indptr[B+1] (absolute offsets into indices/values), values may be NULL (all ones). uid0 = global id of row 0 (RNG key).
 * Writes h1 (bf16 [B, ld_h1]) and coef[nnz] = x_ui * rsqrt(max(|x_u|^2,1e-12)) * mask/keep at the same offsets as indices.
 * Rows longer than 128 nonzeros are split over several CTAs: max_row_nnz bounds the row length of this call, pre_ws
 * (fp32 [B, H]) and counters (int32 [B]) are zero-initialised workspaces that the kernel leaves zeroed again.
 * Optional (training): xc_bf16 [B, ld_xc] (zeroed by the caller) receives coef at column slot_of_item[item] -- the dense
 * coefficient matrix over the batch's active items, i.e. the A operand of the encoder weight-gradient GEMM
 * dW_q0[active] = Xc^T dh1pre (autodiff of MultiVAE.py:152).
 * Optional work list (NULL: a 2-D grid of B x ceil(max_row_nnz/128) CTAs, most of which exit at once when few rows are long):
 * work[n_work], one entry (chunk << 20 | row) per non-empty 128-nonzero chunk of every row (rows without interactions: chunk 0),
 * so the grid holds exactly the chunks that exist; B < 2^20.                                                                     */
int ltg_enc_gather_fwd(const int32_t* indptr, const int32_t* indices, const float* values, int B, int n_items, int64_t uid0,
                       const void* W_enc_bf16, const float* b_q0, float keep, uint64_t seed, uint32_t step,
                       const uint32_t* step_dev, void* h1_bf16, int ld_h1, float* coef, int max_row_nnz, float* pre_ws,
                       int32_t* counters, const int32_t* slot_of_item, void* xc_bf16, int ld_xc, const int32_t* work, int n_work,
                       void* stream);

/* Catalog-sharded layout (SURVEY 8e, config X): the same gather-sum over THIS rank's item shard. indices hold shard-local item ids
 * (rows of W_shard), item_offset + id is the global id (dropout key), n_items_global the whole catalog; row_rnorm[B] =
 * rsqrt(|x_u|^2) over the user's whole row. The fp32 partial pre-activation is ADDED into pre_sum [B, H] (zeroed by the caller); the
 * ranks all-reduce pre_sum and finish with ltg_bias_tanh. coef / xc as in ltg_enc_gather_fwd.                                     */
int ltg_enc_gather_partial(const int32_t* indptr, const int32_t* indices, int B, int n_items_global, int item_offset, int64_t uid0,
                           const void* W_shard_bf16, const float* row_rnorm, float keep, uint64_t seed, uint32_t step,
                           const uint32_t* step_dev, float* pre_sum, float* coef, int max_row_nnz, const int32_t* slot_of_item,
                           void* xc_bf16, int ld_xc, void* stream);
/* out = bf16(tanh(pre + bias)) row-wise, N % 4 == 0 (MultiVAE.py:152-155 after the cross-shard sum).                               */
int ltg_bias_tanh(const float* pre, int ld, const float* bias, int B, int N, void* out_bf16, int ld_out, void* stream);

/* Data-parallel encoder gradient: rebuilds the forward coefficients of the GLOBAL batch's interactions that fall into this
 * rank's item shard (entry e: global batch row e_row[e], item e_item[e], shard slot e_slot[e]; row_uid / row_rnorm per global
 * row) and scatters them into xc_bf16[row, slot] (zeroed by the caller). The dropout bits are recomputed, not communicated.  */
int ltg_enc_coef_scatter(const int32_t* e_row, const int32_t* e_item, const int32_t* e_slot, const int64_t* row_uid,
                         const float* row_rnorm, int n_entries, int n_items, float keep, uint64_t seed, uint32_t step,
                         const uint32_t* step_dev, void* xc_bf16, int ld_xc, void* stream);

/* ---- a3/a4: latent head (MultiVAE.py:157-162,178-181): KL, std, reparameterisation ---------------------------------
 * mulv fp32 [B, 2L] = [mu | logvar]. eps may be NULL (Philox Box-Muller keyed by uid). Writes z bf16 [B, ld_z],
 * zmu fp32 [B, L] = z - mu, adds sum_u KL_u to scal[LTG_S_KL_SUM].                                                    */
int ltg_latent_fwd(const float* mulv, const float* eps, int B, int64_t uid0, float is_training, uint64_t seed, uint32_t step,
                   const uint32_t* step_dev, void* z_bf16, int ld_z, float* zmu, float* scal, void* stream);
/* backward of the above + anneal*KL: dmulv bf16 [B, ld] and bias grad db_q1[2L] (zeroed by caller).
 * anneal is read from scal[LTG_S_ANNEAL] when anneal < 0.                                                              */
int ltg_latent_bwd(const float* dz, const float* mulv, const float* zmu, int B, int B_global, float anneal, const float* scal,
                   void* dmulv_bf16, int ld, float* db_q1, void* stream);

/* Fused middle of the generator (MultiVAE.py:151-162,178-181,168-172), forward: kernel A = [mu|logvar] = h1 W_q1 + b_q1, KL and
 * the reparameterisation; kernel B = h2 = tanh(z W_p0 + b_p0). 16 batch rows x one fifth of the columns per CTA (160 CTAs at
 * B = 500), mma.sync m16n8k16, weights streamed from L2. W_q1 bf16 [600,400], W_p0 bf16 [200,600] row-major. Outputs as
 * ltg_latent_fwd plus h2 (bf16 [B, ld_h2], columns < 600 written). ld_h1 and ld_z multiples of 8.                              */
int ltg_vae_mid_fwd(const void* h1_bf16, int ld_h1, const void* Wq1_bf16, const float* b_q1, const void* Wp0_bf16,
                    const float* b_p0, const float* eps, int B, int64_t uid0, float is_training, uint64_t seed, uint32_t step,
                    const uint32_t* step_dev, float* mulv, void* z_bf16, int ld_z, float* zmu, void* h2_bf16, int ld_h2,
                    float* scal, void* stream);
/* Its backward (autodiff of the same lines) from dh2pre bf16 [B,600] (ltg_tanh_bwd's output): kernel A = dz = dh2pre W_p0^T and
 * the latent backward -> dmulv bf16 [B,400], db_q1[400]; kernel B = dh1 = dmulv W_q1^T, dh1pre = dh1 (1 - h1^2) as fp32 + bf16
 * [B,600], db_q0[600]. Bias gradients are accumulated atomically (zeroed by the caller). The weight gradients (contractions
 * over the batch) stay on ltg_gemm_bf16.                                                                                      */
int ltg_vae_mid_bwd(const void* dh2pre_bf16, const void* Wp0_bf16, const void* Wq1_bf16, const float* mulv, const float* zmu,
                    const void* h1_bf16, int ld_h1, int B, int B_global, float anneal, const float* scal, void* dmulv_bf16,
                    float* dh1pre, void* dh1pre_bf16, float* db_q1, float* db_q0, void* stream);
/* The same two operators on the tcgen05 tensor cores (mid_tc.cu): one launch each, a CTA owns 128 batch rows and chains both GEMMs
 * through TMEM / shared memory; identical arguments and results (bf16 operands, fp32 accumulate).                               */
int ltg_vae_mid_fwd_tc(const void* h1_bf16, int ld_h1, const void* Wq1_bf16, const float* b_q1, const void* Wp0_bf16,
                       const float* b_p0, const float* eps, int B, int64_t uid0, float is_training, uint64_t seed, uint32_t step,
                       const uint32_t* step_dev, float* mulv, void* z_bf16, int ld_z, float* zmu, void* h2_bf16, int ld_h2,
                       float* scal, void* stream);
int ltg_vae_mid_bwd_tc(const void* dh2pre_bf16, const void* Wp0_bf16, const void* Wq1_bf16, const float* mulv, const float* zmu,
                       const void* h1_bf16, int ld_h1, int B, int B_global, float anneal, const float* scal, void* dmulv_bf16,
                       float* dh1pre, void* dh1pre_bf16, float* db_q1, float* db_q0, void* stream);

/* dx = dy * (1 - y^2) for y = tanh(.) stored as bf16 [B, ld_y]; outputs bf16 and/or fp32; column sums -> dbias (atomic).
 * dy may be given as n_partials split-K partial buffers (dy + s*partial_stride), which are summed on the fly.             */
int ltg_tanh_bwd(const float* dy, int ld_dy, int n_partials, int64_t partial_stride, const void* y_bf16, int ld_y, int B, int N,
                 void* dx_bf16, int ld_dxb, float* dx_f32, int ld_dxf, float* dbias, void* stream);

/* ---- a5/a6: decoder + catalog softmax (MultiVAE.py:169,108-112,143) -------------------------------------------------
 * logits = h2 * W_dec + b_dec through the tcgen05 GEMM with the softmax-statistics epilogue: bf16 logits stash
 * [B, ld_logits] (NULL = statistics only) and partial (max,sumexp) pairs: partial[n_blocks][B] float2 with
 * n_blocks = ltg_dec_logits_nblk(B, n_items) = 4 x the number of column tiles the launch uses for this shape (the tile width is
 * chosen per shape against wave quantisation; never more than 4*ceil(n_items/128) rows). The row passes below take n_blocks.
 * partial may be NULL when only the logits are wanted (phase A, train.py:200: the sampler needs no normaliser).                */
int ltg_dec_logits_nblk(int B, int n_items);
int ltg_dec_logits_fwd(const void* h2_bf16, int ld_h2, const void* WdT_bf16, const float* b_dec, int B, int n_items,
                       void* logits_bf16, int ld_logits, float* partial, void* stream);
/* Row pass: lse[B]; nll: scal[NLL_SUM] += -sum_i x_ui (logit_ui - lse_u); sampled-probability sum per user s_u[B] and
 * scal[SUM_P] (train.py:145-149). samp_* may be NULL (VAE-only / evaluation). xw[B] = sum_i x_ui.                       */
int ltg_dec_row_stats(const float* partial, int n_blocks, const void* logits_bf16, int ld_logits, int B,
                      const int32_t* indptr, const int32_t* indices, const float* values,
                      const int32_t* samp_ptr, const int32_t* samp_items, const int32_t* samp_valid,
                      float* lse, float* xw, float* s_u, float* scal, void* stream);
/* softmax probabilities (generator_out, MultiVAE.py:143) materialised as fp32 [B, ld_out] -- compatibility path only. */
int ltg_dec_probs(const void* logits_bf16, int ld_logits, const float* lse, int B, int n_items, float* out, int ld_out, void* stream);
/* d g_loss / d logits (train.py:155 + MultiVAE.py:110-119 under autodiff), Appendix A of SURVEY.md:
 *   dl_ui = pi_ui (xw_u/Bg + lam*Ybar*s_u) - x_ui/Bg - lam*Ybar*pi_ui*m_ui,  Ybar = scal[SUM_Y]/scal[CNT]
 * dense pass then sparse fix-ups; bf16 [B, ld]. lam = GANLAMBDA (0 disables the adversarial term).                     */
int ltg_dec_dlogits(const void* logits_bf16, int ld, const float* lse, const float* xw, const float* s_u, int B, int n_items,
                    int B_global, float lam, const float* scal,
                    const int32_t* indptr, const int32_t* indices, const float* values,
                    const int32_t* samp_ptr, const int32_t* samp_items, const int32_t* samp_valid,
                    void* dl_bf16, void* stream);

/* Fused G-step variant of ltg_dec_row_stats + ltg_dec_dlogits: one CTA per user computes lse / NLL / sampled-probability sum and
 * writes its row of d g_loss / d logits (dense part + sparse fix-ups). scal[SUM_Y], scal[CNT] must be final before the call.     */
int ltg_dec_row_bwd(const float* partial, int n_blocks, const void* logits_bf16, int ld, int B, int n_items, int B_global, float lam,
                    const int32_t* indptr, const int32_t* indices, const float* values,
                    const int32_t* samp_ptr, const int32_t* samp_items, const int32_t* samp_valid,
                    float* lse, float* scal, void* dl_bf16, void* stream);

/* ---- a13: TF-semantics Adam (train.py:160-164; F6 shared step, F7 dense) ------------------------------------------
 * p,m,v fp32 updated in place; g fp32; optional bf16 shadow with the same layout. lr_t < 0: read scal[LTG_S_LR_T].
 * g may be given as n_partials buffers (g + s*partial_stride: split-K partials of the weight-gradient GEMMs), summed on the fly. */
int ltg_adam(float* p, float* m, float* v, const float* g, int n_partials, int64_t partial_stride, void* shadow_bf16, int64_t n,
             float lr_t, const float* scal, float beta1, float beta2, float eps, void* stream);
/* Weight-gradient GEMM with the optimizer step as its epilogue (decoder W_p1^T, single GPU): G[M,N] = A^T B with A bf16 stored
 * [K, lda >= M] and B bf16 stored [K, ldb >= N] (for the decoder: A = dlogits [B, I], B = [h2 | 1] [B, 601]); for columns
 * < n_cols the accumulator is the complete gradient and ltg_adam's update is applied to p/m/v fp32 [M, ld] and the bf16 shadow
 * in place, so the fp32 gradient matrix is never written; column aux_col (bias gradient) goes to aux_out[M]. train.py:163-164. */
int ltg_wgrad_adam(const void* A, int lda, const void* B, int ldb, int M, int N, int K, float* p, float* m, float* v, void* shadow_bf16,
                   int ld, int n_cols, int aux_col, float* aux_out, float lr_t, const float* scal, float beta1, float beta2, float eps,
                   void* stream);

/* ---- e: data-parallel exchange over NVLink peer memory (one node; SURVEY 8e) ------------------------------------------
 * Every table argument is a HOST array of `world` (<= 8) device pointers, entry r = rank r's instance of a peer-mapped buffer
 * (CUDA VMM / symmetric memory set up by the caller; entry `rank` is the local one). `pads` = peer-mapped uint32
 * [LTG_PEER_SLOTS][8] signal words, zero-initialised; `epochs` = local device uint32[LTG_PEER_SLOTS], zero-initialised.
 * All ranks must issue the same sequence of barrier-carrying calls per slot; one slot per stream that issues them.
 * `*_mc` arguments: the NVLS multicast address of the same buffer (NULL = unicast loads/stores to every table entry): stores
 * are replicated and gradient loads are summed inside the NVSwitch (multimem.st / multimem.ld_reduce).                     */
#define LTG_PEER_SLOTS 4
/* every rank has executed all work ordered before this call on its stream (and its peer writes are visible) */
int ltg_peer_barrier(void* const* pads, int rank, int world, int slot, uint32_t* epochs, void* stream);
/* in-place all-reduce (sum, rank order) of floats [offset, offset+count), count <= 1024, in one single-CTA kernel */
int ltg_peer_allreduce_small(void* const* bufs, int64_t offset, int count, void* const* pads, int rank, int world, int slot,
                             uint32_t* epochs, void* stream);
/* out[i] = sum_r bufs[r][offset + i], i < n; `out` must not be one of the peer-visible buffers; caller orders it with barriers */
int ltg_peer_reduce(void* const* bufs, const float* bufs_mc, int64_t offset, int64_t n, int world, float* out, void* stream);
/* copy `bytes` from src to byte offset dst_offset_bytes of every rank's dst buffer (all-gather by pushing; 16-byte granularity) */
int ltg_peer_push(const void* src, int64_t bytes, void* const* dst, void* dst_mc, int64_t dst_offset_bytes, int world, void* stream);
/* ltg_adam over this rank's shard p/m/v[n] = elements [offset, offset+n) of the full tensor, with the reduce-scatter and the
 * all-gather fused in: g = sum_r grads[r][offset+i] (fp32, read from every rank), bf16(p) stored to shadows_bf16[r][offset+i]
 * of every rank. offset and n multiples of 4.                                                                            */
int ltg_adam_peer(float* p, float* m, float* v, void* const* grads, const float* grads_mc, void* const* shadows_bf16, void* shadows_mc,
                  int64_t offset, int64_t n, int world, float lr_t, const float* scal, float beta1, float beta2, float eps, void* stream);

/* ltg_enc_adam over this rank's item rows (p/m/v = shard base, slot_of_item = shard-local table) with the all-gather fused in:
 * the updated bf16 row is stored at element offset `offset` + local index of every rank's encoder shadow.                   */
int ltg_enc_adam_peer(float* p, float* m, float* v, void* const* shadows_bf16, void* shadows_mc, int64_t offset, int n_items,
                      const int32_t* slot_of_item,
                      const float* G, int world, float lr_t, const float* scal, float beta1, float beta2, float eps, void* stream);

/* Encoder weight W_q0 [n_items, H]. Its gradient X^T dh1pre is non-zero only on the batch's ACTIVE items, so it is built
 * compactly: G[slot, :] = sum over the item's batch entries of coef * dh1pre[row, :], one CTA per active item
 * (act_ptr[n_active+1] delimits the item's entries in csc_row[] = batch row / csc_pos[] = offset into coef).                */
int ltg_enc_wgrad_compact(float* G, int n_active, const int32_t* act_ptr, const int32_t* csc_row, const int32_t* csc_pos,
                          const float* coef, const float* dh1pre, int ld_dh1, void* stream);
/* Dense TF-Adam sweep over W_q0 (every row moves, F7); row i takes gradient G[slot_of_item[i], :] (slot -1: zero).
 * rows: 0 = every row; 1 = only the rows with slot -1 (zero gradient: needs nothing from the backward pass, so the engine
 * issues it at the start of the G step); 2 = only the batch's active rows.                                                    */
int ltg_enc_adam(float* p, float* m, float* v, void* shadow_bf16, int n_items, const int32_t* slot_of_item, const float* G,
                 float lr_t, const float* scal, float beta1, float beta2, float eps, int rows, void* stream);
/* out[i] = sum over s < n_partials of src[s * stride + i] (n, stride multiples of 4): split-K partials -> one gradient buffer.   */
int ltg_sum_partials(const float* src, int n_partials, int64_t stride, int64_t n, float* out, void* stream);
/* Data parallel: zeroes the entries ltg_enc_coef_scatter wrote (same e_row / e_slot arrays) once the shard GEMM has read them.   */
int ltg_enc_coef_clear(const int32_t* e_row, const int32_t* e_slot, int n_entries, void* xc_bf16, int ld_xc, void* stream);
/* Restores the all-zero state of the dense coefficient matrix xc[B, ld_xc] that ltg_enc_gather_fwd filled for the batch rows
 * indptr[0..B] (train.py:194-198 made this matrix dense on the host): one store per interaction. nnz_hint sizes the grid.   */
int ltg_enc_xc_clear(const int32_t* indptr, const int32_t* indices, int B, int nnz_hint, const int32_t* slot_of_item, void* xc_bf16,
                     int ld_xc, void* stream);
/* Dense gradient of W_q0 (parity checks / data-parallel all-reduce path): dW[i, :] = G[slot_of_item[i], :] or 0.             */
int ltg_enc_wgrad_expand(float* dW, int n_items, const int32_t* slot_of_item, const float* G, void* stream);

/* ---- a9/a10: niche sampling + pair construction (sample.py:40-67, train.py:212-251) --------------------------------
 * Per user u: candidates cand[cand_ptr[u]..), draw n_u = samp_ptr[u+1]-samp_ptr[u] items without replacement with
 * probability proportional to softmax(logits)[u, cand] (Gumbel-top-k == numpy's successive draw in distribution, F9),
 * emit them in ascending item order at slots samp_ptr[u].., each paired with a uniformly drawn popular item of the user
 * (pop_ptr/pop_items), valid[slot] = +1 if both ids are in the item-feature table (item_valid[n_items] bytes, F10), else -1.
 * *cnt (int32, may be NULL) += number of valid pairs. user_order (may be NULL): permutation of the batch rows giving the CTA
 * launch order (heaviest candidate lists first).                                                                            */
int ltg_sample_pairs(const void* logits_bf16, int ld_logits, int B, int n_items, int64_t uid0,
                     const int32_t* cand_ptr, const int32_t* cand_items, const int32_t* samp_ptr,
                     const int32_t* pop_ptr, const int32_t* pop_items, const uint8_t* item_valid,
                     uint64_t seed, uint32_t step, const uint32_t* step_dev,
                     int32_t* samp_items, int32_t* samp_partner, int32_t* samp_valid, int32_t* cnt, int max_cand,
                     const int32_t* user_order, void* stream);
/* Same, with the candidates' logits given explicitly (cand_vals[j] belongs to cand_items[j]; catalog-sharded layout: every rank
 * contributes the logits of the candidates it owns and the sum is all-reduced); logits_bf16 may then be NULL.                 */
int ltg_sample_pairs_vals(const void* logits_bf16, int ld_logits, const float* cand_vals, int B, int n_items, int64_t uid0,
                          const int32_t* cand_ptr, const int32_t* cand_items, const int32_t* samp_ptr,
                          const int32_t* pop_ptr, const int32_t* pop_items, const uint8_t* item_valid,
                          uint64_t seed, uint32_t step, const uint32_t* step_dev,
                          int32_t* samp_items, int32_t* samp_partner, int32_t* samp_valid, int32_t* cnt, int max_cand,
                          const int32_t* user_order, void* stream);

/* ---- a11/a12: discriminator (discriminator.py:14-55, train.py:142) --------------------------------------------------
 * Frozen embedding gather (F5): rows of E_bf16 [n_items, 128] (cols 100.. are zero) -> Xp, Xn bf16 [P, 128].            */
int ltg_disc_gather(const void* E_bf16, const int32_t* pop_ids, const int32_t* niche_ids, int P, void* Xp, void* Xn, void* stream);
/* The whole forward of discriminator.py:16-55 on P gathered pairs as one tcgen05 kernel per 128 pairs (branch layers, fc1 and
 * the head chained through TMEM / shared memory), replacing three ltg_gemm_bf16 launches + ltg_disc_head with identical dropout
 * masks (streams rng_stream, +1, +2). Weights in the ones-row layout of the package's discriminator module: W1 [k1, ld1],
 * W2 [k1, ld2], W3 [k3, ld3] bf16 row-major (bias = row k1-1 / row one3). Writes the hidden activation Hd bf16 [P, k3]
 * (columns [0,off2) branch 1, [off2, off2+h2) branch 2, one3 = 1), y[P], the scal / dz3 / dw4 / db4 outputs of ltg_disc_head
 * (dz3 bf16 [P, ld3], NULL = forward only). dz12_bf16 (optional, needs dz3): the backward continues in the same tile with
 * dz12 [P, k3] = (dz3 W3^T) * d/da dropout(tanh(a)) recovered from Hd (autodiff of discriminator.py:25-44 under train.py:163), so
 * the separate backward GEMM is not needed. ltg_disc_fused_supported tells whether the sizes fit the kernel's fixed tiles.
 * rng_row0: dropout-counter row of this launch's pair 0. A launch over pairs [r, r + P) of a larger batch (pointers advanced to
 * row r) with rng_row0 = r draws exactly the masks the one launch over the whole batch draws for those rows (engine.run_step runs
 * the real pairs of the D update, which do not depend on phase A, beside phase A, and the generated pairs behind the sampler).   */
/* debug: device buffer (148*2*32 u64) that receives per-phase globaltimer stamps of the following launches; NULL switches it off */
int ltg_disc_fused_set_trace(void* buf);
int ltg_disc_fused_supported(int k1, int ld1, int ld2, int ld3, int off2, int one3, int h2, int k3);
int ltg_disc_fwd_fused(const void* Xp_bf16, const void* Xn_bf16, int P, int k1, const void* W1_bf16, int ld1, const void* W2_bf16, int ld2,
                       int h2, const void* W3_bf16, int ld3, int k3, int off2, int one3, const float* w4, const float* b4,
                       const int32_t* label, float keep, uint64_t seed, uint32_t rng_stream, uint32_t rng_step,
                       const uint32_t* rng_step_dev, void* Hd_bf16, float* y, float* scal, void* dz3_bf16, float* dw4, float* db4,
                       void* dz12_bf16, int rng_row0, void* stream);
/* Head: s = Y3*w4 + b4, y = sigmoid(s); label[row]: 0 real, 1 generated, <0 ignored.
 * Accumulates scal[D_LOSS], scal[SUM_Y] and scal[CNT] (generated rows), and when dz3 != NULL the backward seed:
 * dz3 bf16 [P, ld] = ds*w4*dact(Y3), dw4[h3] += Y3^T ds, *db4 += sum ds. (The fc1 bias gradient comes out of the
 * weight-gradient GEMM through the ones column of the hidden activation.)                                              */
int ltg_disc_head(const void* Y3_bf16, int ld, int P, int h3, const float* w4, const float* b4, const int32_t* label,
                  float keep, float* y_out, float* scal, void* dz3_bf16, float* dw4, float* db4, void* stream);
/* ---- a16/a17: ranking metrics (eval_functions.py:11-62, train.py:341) -----------------------------------------------
 * Per row: scores (fp32 or bf16, pitch ld) with the row's seen items (seen_ptr/seen_items, may be NULL) forced to -inf,
 * exact top-k (k <= 128; ties: lowest index first) sorted by score descending -> topk_idx [n, k] (may be NULL),
 * dcg[n] (fp64, as the reference's NumPy) = sum_{r<k} held(top_r)/log2(r+2), hits[n, n_rk] = |top-rk[j] AND heldout| for up to 4 recall cut-offs rk[j] <= k.
 * held_ptr/held_items: CSR of the held-out interactions (sorted within row).                                            */
int ltg_topk_metrics(const void* scores, int is_bf16, int64_t ld, int n_rows, int n_items,
                     const int32_t* seen_ptr, const int32_t* seen_items, const int32_t* held_ptr, const int32_t* held_items,
                     int k, const int32_t* rk_host, int n_rk, int32_t* topk_idx, double* dcg, int32_t* hits, void* stream);
/* Long-tail evaluation: ltg_topk_metrics (same arguments, same lists, bit-identical topk_idx / dcg / hits, same staged / streaming
 * choice) plus, per row, from the same sorted list of kk = min(k, n_items) items: dcg_niche[n] (fp64) = sum over listed held-out NICHE
 * items of 1/log2(r+2), hits_niche[n, n_rk] = |top-rk[j] AND heldout AND niche|, n_niche_top[n] = |list AND niche|, pop_sum[n] = sum of
 * item_pop over the list. niche_bits: (n_items+31)/32 words, bit i%32 of word i/32 set for a niche item (the allow_bits format of
 * ltg_topk_recommend); item_pop [n_items]: training interactions per item. rec_count [n_items] += 1 for every listed item of every row
 * with a non-empty held-out set: it is NOT cleared, so it accumulates across launches (zero it before the first). Every pointer is
 * required except seen_ptr / seen_items and topk_idx (may be NULL, as for ltg_topk_metrics) and rk_host / hits when n_rk == 0.       */
int ltg_topk_longtail(const void* scores, int is_bf16, int64_t ld, int n_rows, int n_items,
                      const int32_t* seen_ptr, const int32_t* seen_items, const int32_t* held_ptr, const int32_t* held_items,
                      int k, const int32_t* rk_host, int n_rk, int32_t* topk_idx, double* dcg, int32_t* hits,
                      const uint32_t* niche_bits, const int32_t* item_pop, double* dcg_niche, int32_t* hits_niche, int32_t* n_niche_top,
                      int64_t* pop_sum, int32_t* rec_count, void* stream);
/* Recommendation lists. Per row u of fp32 logits (pitch ld; columns n_items..ld are never read), an item is ELIGIBLE when it is not in
 * seen_items[seen_ptr[u] .. seen_ptr[u+1]) and its bit of allow_bits ((n_items+31)/32 words, bit i%32 of word i/32) is set. Excluded
 * items are never listed. out_idx [n, k]: the min(k, #eligible) eligible items with the highest logits ordered by (logit desc, item id
 * asc), the tie rule of ltg_topk_metrics; remaining slots -1. out_logit [n, k]: the listed logits, bit-equal to the input, -inf for
 * padding. out_lse [n]: log sum_i exp(logit_i) over ALL n_items columns whatever the filters exclude (max-shifted, fp32, expf), so
 * out_prob [n, k] (may be NULL) = exp(logit - lse) is the generator's softmax probability (MultiVAE.py:143), 0 for padding.
 * 1 <= k <= 128. Rows of at most 49,152 items with 16-byte aligned rows are staged in shared memory; larger catalogs stream.        */
int ltg_topk_recommend(const float* scores, int64_t ld, int n_rows, int n_items,
                       const int32_t* seen_ptr, const int32_t* seen_items,   /* may both be NULL: nothing excluded */
                       const uint32_t* allow_bits,                           /* may be NULL: every item allowed   */
                       int k, int32_t* out_idx, float* out_logit, float* out_prob, float* out_lse, void* stream);

/* ---- a1 / f3: dataset ingestion on the host cores (data_processing.py:6-37: pandas.read_csv + scipy csr_matrix) -----------
 * HOST entry points (no kernels, no stream): every pointer below is a host pointer.
 * ltg_csv_open: memory-maps the CSV at `path_host`, finds the columns named `row_name_host` / `col_name_host` in its header line
 * (tp['uid'], tp['sid'] at data_processing.py:8-15; further columns are ignored), parses the integer ids with n_threads threads
 * (<= 0: all cores) and returns an opaque handle in *handle_host. stats_host (may be NULL) receives
 * [n_pairs, row_min, row_max, col_min, col_max] -- what load_train_data / load_tr_te_data derive their shapes and uid offset from
 * (uid.max() + 1, uid.min(); min/max over both files).
 * ltg_csv_pairs: the parsed pairs in file order (load_user_items, data_processing.py:72-96), n_pairs int64 each.
 * ltg_csv_to_csr: CSR of the pair list as scipy's csr_matrix((ones, (rows - row_offset, cols)), shape=(n_rows, n_cols)) followed by
 * sort_indices builds it: duplicates summed into counts_host, column ids ascending within a row. indptr_host [n_rows + 1];
 * indices_host / counts_host hold n_pairs entries (capacity), *nnz_host of them are written. An id outside the shape is an error.
 * ltg_csv_close: frees the handle.                                                                                          */
int ltg_csv_open(const char* path_host, const char* row_name_host, const char* col_name_host, int n_threads, void** handle_host,
                 int64_t* stats_host);
int ltg_csv_pairs(void* handle_host, int64_t* rows_host, int64_t* cols_host);
int ltg_csv_to_csr(void* handle_host, int64_t row_offset, int64_t n_rows, int64_t n_cols, int n_threads, int32_t* indptr_host,
                   int32_t* indices_host, float* counts_host, int64_t* nnz_host);
int ltg_csv_close(void* handle_host);

/* ---- f1: GAN side tables on the host cores (data_processing.py:170-271) ------------------------------------------------
 * HOST entry points. The overlap coefficients (data_processing.py:100-167) are read from the sparse co-occurrence counts
 * C = X^T X: CSR with int64 row pointers, column ids sorted within a row (int32, or int64 when indices_are_64), int64 counts, and
 * deg[i] = C[i,i]; overlap(a,b) = C[a,b] / min(deg[a], deg[b]) in float64, 0 where an item never occurs. Users are given as ragged
 * lists in file order: un_ptr/un_items the niche items, up_ptr/up_items the popular items (load_user_items, 72-96); eligible[u] =
 * the user appears in both (train.py:213-217).
 * ltg_cand_sets = load_items_to_sample (170-224): per eligible user the own niche items plus the top max(2n, 10-n) other items of
 * niche_sorted (ascending ids) by their best overlap with any own niche item (ties: ascending id), written sorted to
 * out_items[out_ptr[u] ...] with the count in out_count[u]; out_ptr must reserve n + max(2n, 10-n) entries per user.
 * ltg_real_pairs = load_vectors (227-271): per eligible user and niche item the user's popular item with the highest overlap (first
 * maximum in list order), kept when both ids are valid (item_valid, = membership in ITEM_FEATURE_DICT, 258-262); pairs of user u
 * are written from position un_ptr[u] of out_niche / out_pop, their number to out_count[u].                                  */
int ltg_cand_sets(const int64_t* C_indptr_host, const void* C_indices_host, int indices_are_64, const int64_t* C_counts_host,
                  const double* deg_host, int n_items, const int32_t* niche_sorted_host, int n_niche, const int64_t* un_ptr_host,
                  const int32_t* un_items_host, const uint8_t* eligible_host, int64_t n_users, int n_threads,
                  const int64_t* out_ptr_host, int32_t* out_items_host, int32_t* out_count_host);
int ltg_real_pairs(const int64_t* C_indptr_host, const void* C_indices_host, int indices_are_64, const int64_t* C_counts_host,
                   const double* deg_host, int n_items, const uint8_t* item_valid_host, const int64_t* un_ptr_host,
                   const int32_t* un_items_host, const int64_t* up_ptr_host, const int32_t* up_items_host,
                   const uint8_t* eligible_host, int64_t n_users, int n_threads, int32_t* out_niche_host, int32_t* out_pop_host,
                   int32_t* out_count_host);

/* ---- misc ------------------------------------------------------------------------------------------------------------ */
/* fp32 -> bf16 with optional re-pitch: dst[r*ld_dst + c] = src[r*ld_src + c]                                             */
int ltg_cast_bf16(const float* src, int64_t ld_src, void* dst, int64_t ld_dst, int64_t rows, int64_t cols, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* LTGAN_H_ */
