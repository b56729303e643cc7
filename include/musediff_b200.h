/*
 * musediff_b200 — C-ABI of the B200-native MuseDiffusion reverse-diffusion sampling path.
 *
 * The reference (YAIxPOZAlabs/MuseDiffusion) has no FFI of its own: its boundary is the Python call surface
 * exercised by MuseDiffusion/run/sample.py (SURVEY.md section 8b).  These entry points are what a ctypes binding
 * placed behind that surface calls; each cites the reference code it replaces (paths relative to the reference
 * root).  Conventions: plain device pointers + sizes, no torch types, no allocation, no internal threads, work is
 * enqueued on the caller's `stream`; return 0 (MD_OK) or a negative code, text via md_last_error().
 * All tensors are contiguous row-major; "M" is the token count B*L.
 */
#ifndef MUSEDIFF_B200_H
#define MUSEDIFF_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#ifndef __CUDA_RUNTIME_H__
typedef struct CUstream_st* cudaStream_t;
#endif

#define MD_OK 0
#define MD_ERR_ARG (-1)
#define MD_ERR_CUDA (-2)

/* epilogues of md_linear_bf16 */
#define MD_EPI_BIAS 0          /* y = xW^T + b                                                           */
#define MD_EPI_BIAS_GELU 1     /* erf-GELU(y)            HF BertIntermediate (called from network.py:151) */
#define MD_EPI_BIAS_TANH 2     /* tanh(y)                input_up_proj / output_down_proj, network.py:69-70,83-84 */
/* (3 is reserved: the residual add of HF BertSelfOutput / BertOutput is fused into md_layernorm_bf16 instead) */
#define MD_EPI_BIAS_POS_TIME 4 /* y + pos[l] + temb[b]   network.py:146-148 pre-LayerNorm sum            */
#define MD_EPI_BIAS_SPLIT 5    /* out = bf16 [M, 2N] = [hi | lo] of y (hi = bf16(y), lo = bf16(y - hi)): the last Linear of
                                * output_down_proj (network.py:85) feeding md_round_argmin_tc without an fp32 round trip */

/* modes of md_posterior_step */
#define MD_STEP_DDPM 0 /* GaussianDiffusion.p_sample,    models/diffusion.py:349-404 */
#define MD_STEP_DDIM 1 /* GaussianDiffusion.ddim_sample, models/diffusion.py:701-757 */

#define MD_MAX_CONST_T 2048 /* schedules up to this length live in __constant__ memory */

const char* md_last_error(void);
int md_abi_version(void);

/* ---- schedule tables: GaussianDiffusion.__init__ (models/diffusion.py:136-185) + _extract_into_tensor (:904-917).
 * `tables` = 9 host arrays of T floats each (float64 tables already cast to fp32 exactly as diffusion.py:914 does):
 *   0 posterior_mean_coef1   1 posterior_mean_coef2   2 model_log_variance (fixed-large, :313-317)
 *   3 sqrt_recip_alphas_cumprod   4 sqrt_recipm1_alphas_cumprod   5 alphas_cumprod   6 alphas_cumprod_prev
 *   7 sqrt_alphas_cumprod    8 sqrt_one_minus_alphas_cumprod
 * Uploads them to device memory (and rows 0..6 to __constant__ memory when T <= MD_MAX_CONST_T). */
int md_set_schedule(const float* tables, int T, cudaStream_t stream);

/* ---- elementwise / small kernels ---- */
/* fp32 -> bf16 cast of the state x_t (A operand of the first Linear).  n elements. */
int md_cast_f32_bf16(const float* in, void* out_bf16, int64_t n, cudaStream_t stream);
/* The same for fp32 [rows, D] into bf16 rows of stride ld >= D (the padded width Dp of the tensor-core operands, see
 * md_embed_split_padded); columns D..ld-1 are not written.  D and ld multiples of 4. */
int md_cast_f32_bf16_ld(const float* in, void* out_bf16, int64_t rows, int D, int ld, cudaStream_t stream);
/* Models with hidden_dim == encoder hidden size have no input_up_proj / output_down_proj (models/network.py:67-72, 81-86):
 * md_add_pos_time: out[m, :] = bf16((pos[m % L, :] + x[m, :]) + temb[(m / L) * temb_stride, :])  — the pre-LayerNorm sum of
 *   network.py:146-148 taken from the fp32 state itself (emb_x = x, :143-144);  x fp32 [M, H], pos fp32 [L, H].
 * md_cast_bf16_f32: the last hidden state as the fp32 model output (h.type(x.dtype), :155-157).  n elements. */
int md_add_pos_time(const float* x, const float* pos, const float* temb, int temb_stride, int L, int H, void* out_bf16, int64_t M,
                    cudaStream_t stream);
int md_cast_bf16_f32(const void* in_bf16, float* out, int64_t n, cudaStream_t stream);
/* TransformerNetModel.get_embeds (models/network.py:88-89): out[m, :] = E[ids[m], :].  ids int32 or int64. */
int md_embed_gather(const float* E, const void* ids, int ids_is_i64, float* out, int64_t M, int V, int D,
                    cudaStream_t stream);
/* timestep_embedding + time_embed MLP (models/network.py:108-129, 60-65, 139):
 * out[b, :] = W2 silu(W0 [cos(t f), sin(t f)] + b0) + b2, fp32 throughout.  t is the float fed to the model. */
int md_timestep_mlp(const float* t, const float* W0, const float* b0, const float* W2, const float* b2, float* out,
                    float* hidden_ws /* [B, mid_dim] scratch */, int B, int t_dim, int mid_dim, int out_dim,
                    cudaStream_t stream);
/* out = LayerNorm(in + resid) over the last dim of bf16 [M, H] tensors, fp32 statistics (network.py:149 and the HF
 * BertSelfOutput / BertOutput `LayerNorm(dense(x) + input)`, eps = 1e-12).  resid may be NULL.  H must be a multiple
 * of 256 and <= 2048. */
int md_layernorm_bf16(const void* in_bf16, const void* resid_bf16, const float* gamma, const float* beta, float eps,
                      void* out_bf16, int64_t M, int H, cudaStream_t stream);

/* ---- dense contractions (tcgen05 / TMEM / TMA) ---- */
/* nn.Linear with fused epilogue: out[M,N] = epi(A[M,K] W[N,K]^T + bias).  A, W bf16; bias/pos/temb fp32;
 * out bf16 (out_is_f32 = 0) or fp32.  pos: [L,N], temb: [M/L or 1, N] with row stride temb_stride (0 = one shared
 * row) (MD_EPI_BIAS_POS_TIME).  K, N multiples of 8; A, W, out 16-byte aligned. */
int md_linear_bf16(const void* A, const void* W, const float* bias, void* out, int M, int N, int K, int epilogue,
                   int out_is_f32, const float* pos, const float* temb, int temb_stride, int L, cudaStream_t stream);
/* md_linear_bf16 storing only the first out_cols <= N columns: out is [M, out_cols] (row stride out_cols, a multiple of
 * 4 for fp32 and of 8 for bf16 output); the rest is computed and dropped.  The last Linear of a model whose width D is
 * zero-padded to Dp writes its D real columns this way.  MD_EPI_BIAS_SPLIT needs out_cols == N. */
int md_linear_bf16_cols(const void* A, const void* W, const float* bias, void* out, int M, int N, int K, int out_cols,
                        int epilogue, int out_is_f32, const float* pos, const float* temb, int temb_stride, int L,
                        cudaStream_t stream);
/* HF BertSelfAttention without mask (called from network.py:151): qkv bf16 [B*L, 3*NH*DH] laid out
 * [q heads | k heads | v heads] per token, q already scaled by 1/sqrt(DH); out bf16 [B*L, NH*DH] = softmax(qk^T) v.
 * DH must be 64. */
int md_attention_bf16(const void* qkv, void* out, int B, int L, int NH, int DH, cudaStream_t stream);

/* ---- rounding / decode ---- */
/* get_efficient_knn (models/rounding.py:21-28): idx[m] = argmin_v clamp(|E_v|^2 + |x_m|^2 - 2 E_v.x_m, 0),
 * lowest v on ties.  x fp32 [M,D], E fp32 [V,D], idx int32 [M]; margin (optional, fp32 [M]) = second-best minus
 * best distance.  D must be a multiple of 4.
 * Non-finite inputs: every id written lies in [0, V).  A NaN key is clamped to 0 by the clamp above, so it ties with an
 * exact hit (lowest v wins); md_logits_argmax never picks a NaN logit, gives a row with no logit above -inf the lowest
 * id whose logit is -inf, and a row whose logits are all NaN id 0 (what torch.argmax gives for an all-NaN row). */
int md_round_argmin(const float* x, const float* E, int32_t* idx, float* margin, int64_t M, int V, int D,
                    cudaStream_t stream);
/* get_logits + argmax (models/network.py:91-93, run/sample.py:219-220): tok[m] = argmax_v (x_m.E_v + bias_v).
 * D must be a multiple of 4. */
int md_logits_argmax(const float* x, const float* E, const float* bias, int32_t* tok, float* margin, int64_t M, int V,
                     int D, cudaStream_t stream);

/* get_logits with logits_mode = 2 (models/network.py:94-104): scores[m, v] = -sqrt(clamp(|E_v|^2 + |x_m|^2 - 2 x_m.E_v, 0)).
 * dot fp32 [M, dot_stride] holds x_m.E_v (from the split-bf16 md_linear_bf16 contraction), esq fp32 [V] = |E_v|^2
 * (md_embed_split), x fp32 [M, D]; out fp32 [M, V]. */
int md_dist_scores(const float* x, const float* dot, const float* esq, float* out, int64_t M, int V, int dot_stride, int D,
                   cudaStream_t stream);

/* Tensor-core versions of the two reductions above (tcgen05, split-bf16 operands x = xh + xl, E = Eh + El with the four
 * partial products accumulated in fp32: fp32-grade scores, the score matrix stays in TMEM).
 *   md_embed_split: once per embedding matrix.  E2 = bf16 [Vp, 2D] = [Eh | El], sqnorm = fp32 [Vp] = |E_v|^2 (+inf on
 *     the Vp - V padding rows), Vp = md_round_tc_padded_vocab(V); E_clamped (optional) = clamp(E, -1, 1), the rows
 *     md_posterior_step gathers when clip_denoised follows the rounding (clip = 2 there).
 *   md_round_argmin_tc: mode 0: idx[m] = argmin_v (cst[v] - 2 x_m.E_v), cst = sqnorm  (rounding.py:21-28; |x_m|^2 is
 *     constant per row, the reference's clamp(dist, 0) only creates ties on bit-exact hits);
 *     mode 1: idx[m] = argmax_v (x_m.E_v + cst[v]), cst = lm_head bias padded with -inf  (network.py:91-93 + argmax).
 *     x2_ws: bf16 [M, 2D] scratch; with x == NULL it must already hold the [hi | lo] split of x (MD_EPI_BIAS_SPLIT) and
 *     the split pass is skipped.  Lowest index wins ties.  D must be a multiple of 64.
 *     Non-finite inputs: NaN keys never win; a row with no key below +inf (any NaN / inf in x_m makes every key NaN;
 *     in mode 1 every logit -inf or NaN) gets idx 0, so every id written lies in [0, V). */
/* fp32 [rows, D] -> bf16 [rows, copies * 2D]: `copies` repetitions of the two-term split [hi | lo], hi = bf16(x),
 * lo = bf16(x - hi)  (operand of the split-bf16 contractions: rounding, decode, get_logits). */
int md_split_bf16(const float* x, void* out_bf16, int64_t rows, int D, int copies, cudaStream_t stream);
int md_round_tc_padded_vocab(int V);
int md_embed_split(const float* E, int V, int D, void* E2, float* sqnorm, float* E_clamped /* optional fp32 [V, D] */,
                   cudaStream_t stream);
int md_round_argmin_tc(const float* x, const void* E2, const float* cst, void* x2_ws, int32_t* idx, float* margin,
                       int64_t M, int V, int D, int mode, cudaStream_t stream);
/* The two entries above for any D that is a multiple of 4, with the bf16 operands zero-padded to the width Dp (a multiple
 * of 64, >= D; the package uses D rounded up to 64): E2 = bf16 [Vp, 2Dp] = [Eh | 0 | El | 0], x2_ws = bf16 [M, 2Dp] =
 * [xh | 0 | xl | 0].  The zero columns leave every dot product and |E_v|^2 unchanged, so ids equal those of the unpadded
 * contraction.  x, E and E_clamped stay fp32 [., D].  With Dp == D these are md_embed_split / md_round_argmin_tc. */
int md_embed_split_padded(const float* E, int V, int D, int Dp, void* E2, float* sqnorm, float* E_clamped,
                          cudaStream_t stream);
int md_round_argmin_tc_padded(const float* x, const void* E2, const float* cst, void* x2_ws, int32_t* idx, float* margin,
                              int64_t M, int V, int D, int Dp, int mode, cudaStream_t stream);

/* ---- the fused per-step posterior update ----
 * x_{t-1} from x_t for mode DDPM (p_sample :349-404 with p_mean_variance :311-347, q_posterior_mean :257-278) or
 * DDIM (ddim_sample :701-757, _predict_eps_from_xstart :201-205):
 *   pred  = idx ? E[idx] : pred_in                      (denoised_fn_round, rounding.py:31-47)
 *   pred  = clip == 1 ? clamp(pred, -1, 1) : pred       (diffusion.py:323-324, AFTER rounding; clip == 2: E already holds
 *                                                        clamp(E, -1, 1) — md_embed_split's E_clamped — nothing left to do)
 *   DDPM: x' = c1[t] pred + c2[t] x_t + [t != 0] exp(0.5 logvar[t]) n
 *   DDIM: eps = (sr[t] x_t - pred)/srm1[t]; sigma = eta sqrt((1-abp)/(1-ab)) sqrt(1-ab/abp);
 *         x' = pred sqrt(abp) + sqrt(1-abp-sigma^2) eps + [t != 0] sigma n
 *   x'   = mask == 0 ? x_start : x'                     (diffusion.py:394-397, 752-755)
 * n = noise[m, d] if noise != NULL, else a counter-based Philox4x32-7 normal keyed by (seed, step_counter, global
 * element index (seq_offset*L + m)*D + d), truncated to |n| <= top_p by inverse-CDF when top_p > 0 (the law the
 * reference's rejection loop :378-385 samples).  t: int32 schedule index, t[b * t_stride] (t_stride 1 = per sequence,
 * 0 = one value for the batch, as inside the loops :516,887).  mask: int32, indexed m*mask_tok_stride + d*mask_d_stride
 * (NULL = no mask).  step_counter_dev (optional): the step counter is read from this device word instead of the argument.
 * Optional outputs: out_bf16 = bf16 copy of x' (next step's GEMM operand), pred_out = processed
 * pred_xstart, mean_out = the mean before noise ("greedy_mean" of p_sample). */
int md_posterior_step(const float* x_t, const int32_t* idx, const float* pred_in, const float* E, const float* noise,
                      uint64_t seed, uint64_t step_counter, int64_t seq_offset, const int32_t* t, int t_stride,
                      const int32_t* mask, int64_t mask_tok_stride, int64_t mask_d_stride, const float* x_start,
                      float* x_out, void* out_bf16, float* pred_out, float* mean_out, int B, int L, int D, int mode,
                      float eta, int clip, float top_p, const uint64_t* step_counter_dev, cudaStream_t stream);
/* md_posterior_step with out_bf16 rows of stride bf16_ld >= D (a multiple of 4): the padded first-GEMM operand of a
 * model whose width is not a multiple of 64.  Columns D..bf16_ld-1 are not written (zero them once).  Noise stays keyed
 * by the logical index (seq_offset*L + m)*D + d. */
int md_posterior_step_ld(const float* x_t, const int32_t* idx, const float* pred_in, const float* E, const float* noise,
                         uint64_t seed, uint64_t step_counter, int64_t seq_offset, const int32_t* t, int t_stride,
                         const int32_t* mask, int64_t mask_tok_stride, int64_t mask_d_stride, const float* x_start,
                         float* x_out, void* out_bf16, int bf16_ld, float* pred_out, float* mean_out, int B, int L, int D,
                         int mode, float eta, int clip, float top_p, const uint64_t* step_counter_dev, cudaStream_t stream);
/* ---- one step of the DPM-Solver++(2M) sampler (Lu et al., "DPM-Solver++", 2022, Algorithm 2: multistep, second order,
 * data prediction) — an addition beyond the reference, which samples with DDPM / DDIM only ----
 *   p    = idx ? E[idx] : pred_in, clipped as in md_posterior_step (clip 0 / 1 / 2 with the same meaning)
 *   (a, b, c0, c1) = coef[row]: row = *cursor - 1 clamped to [0, n_coef - 1] (the cursor as md_step_advance leaves it, so one
 *        captured graph serves every step), or row 0 when cursor is NULL (then n_coef must be 1)
 *   d    = c1 != 0 ? c0 p + c1 q : c0 p,  q = pred_hist[m, d] (the previous evaluation's p; never read where c1 == 0)
 *   pred_hist[m, d] = p                   (in place, after the read)
 *   x'   = a != 0 ? a x_t + b d : b d     (x_t is not read where a == 0: the row (0, 1, 1, 0) writes p itself)
 *   x'   = mask == 0 ? x_start : x'       (mask as md_posterior_step)
 * fp32, every product and sum rounded separately (no FMA contraction).  x_out may alias x_t; out_bf16 (optional) = bf16
 * copy of x' in rows of stride bf16_ld >= D (a multiple of 4), columns D..bf16_ld-1 never written.  pred_hist fp32 [M, D],
 * coef fp32 [n_coef, 4].  D must be a multiple of 4.  The step draws no noise. */
int md_dpm_solver_step(const float* x_t, const int32_t* idx, const float* pred_in, const float* E, float* pred_hist,
                       const float* coef, int n_coef, const int32_t* cursor, const int32_t* mask, int64_t mask_tok_stride,
                       int64_t mask_d_stride, const float* x_start, float* x_out, void* out_bf16, int bf16_ld, int B, int L,
                       int D, int clip, cudaStream_t stream);
/* Loop state on the device, so that ONE captured CUDA graph of a reverse step can be replayed for every index of the
 * loops diffusion.py:508-540 / :878-901 (the reference rebuilds t = th.tensor([i] * B) on the host every iteration):
 * k = *cursor; *t_cur = t_idx[k]; *tm_cur = t_model[k] (the value _WrappedModel feeds the denoiser, :1027-1032);
 * *ctr_cur = ctr_base + k (Philox counter of md_posterior_step's step_counter_dev); *cursor = k + 1.  n = entries. */
int md_step_advance(int32_t* cursor, const int32_t* t_idx, const float* t_model, int n, int32_t* t_cur, float* tm_cur,
                    uint64_t* ctr_cur, uint64_t ctr_base, cudaStream_t stream);
/* x0 = sqrt_recip[t] x_t - sqrt_recipm1[t] eps  (_predict_xstart_from_eps, diffusion.py:194-199), for
 * predict_xstart = False models. */
int md_xstart_from_eps(const float* x_t, const float* eps, const int32_t* t, int t_stride, float* out, int B, int L,
                       int D, cudaStream_t stream);
/* q_sample (diffusion.py:229-255): out = mask==0 ? x0 : sqrt_ab[t] x0 + sqrt_1m_ab[t] n.  t < 0 means "pure
 * noise": out = mask==0 ? x0 : n (the generation-mode initialisation, run/sample.py:190-193).  Noise as above. */
int md_q_sample(const float* x0, const float* noise, uint64_t seed, uint64_t step_counter, int64_t seq_offset,
                const int32_t* t, int t_stride, const int32_t* mask, int64_t mask_tok_stride, int64_t mask_d_stride,
                float* out, void* out_bf16, int B, int L, int D, cudaStream_t stream);
/* md_q_sample with out_bf16 rows of stride bf16_ld >= D, as md_posterior_step_ld. */
int md_q_sample_ld(const float* x0, const float* noise, uint64_t seed, uint64_t step_counter, int64_t seq_offset,
                   const int32_t* t, int t_stride, const int32_t* mask, int64_t mask_tok_stride, int64_t mask_d_stride,
                   float* out, void* out_bf16, int bf16_ld, int B, int L, int D, cudaStream_t stream);
/* standard-normal / truncated-normal fill with the same Philox stream (testing + generation init). */
int md_fill_normal(float* out, int64_t n, uint64_t seed, uint64_t step_counter, int64_t elem_offset, float top_p,
                   cudaStream_t stream);


/* ---- SURVEY.md section 8(f) row 1: token-level half of the post-sampling decode, batched -------------------------
 * What SequenceToMidi.decode does before the MIDI writer (MuseDiffusion/utils/decode_util.py:207-214) for every row of
 * a sampled batch: split_meta_midi (:192-199: meta / note split from the mask), remove_padding (:72-82: cut after the
 * first EOS), restore_chord (:84-141: splice the meta's (position, chord) pairs back in), validate_once (:143-155) and,
 * if strict != 0, validate_rigidly (:157-184).  Replaces the per-row Python of batch_decode_seq2seq /
 * batch_decode_generation (:259-384) up to the point where miditoolkit takes over.
 *   tokens, mask  int32 [B, L] (sampled ids; the ORIGINAL input mask: 0 over meta + first EOS)
 *   status        int32 [B]     MD_DECODE_* below (the reference raises SequenceToMidiError(msg) for 1..4 and lets an
 *                               IndexError escape — aborting the run — for 5)
 *   note_len      int32 [B]     length of the restored note sequence (0 when it does not exist)
 *   notes         int32 [B, 2L] restored note sequence, zero padded
 *   meta          int32 [B, 11] the 11 meta tokens handed to the MIDI writer */
enum {
    MD_DECODE_OK = 0,
    MD_DECODE_NO_EOS = 1,             /* "NO EOS TOKEN" */
    MD_DECODE_RESTORE_FAILED = 2,     /* "RESTORE_CHORD FROM META FAILED" */
    MD_DECODE_VALIDATION_FAILED = 3,  /* "VALIDATION OF SEQUENCE FAILED" */
    MD_DECODE_STRICT_FAILED = 4,      /* "STRICT VALIDATION OF SEQUENCE FAILED" */
    MD_DECODE_INDEX_ERROR = 5,        /* the reference's numpy indexing raises IndexError here */
    MD_DECODE_TOO_LONG = 6            /* restored sequence longer than 2L (degenerate meta; the reference has no bound) */
};
int md_decode_prepare(const int32_t* tokens, const int32_t* mask, int B, int L, int strict, int32_t* status,
                      int32_t* note_len, int32_t* notes, int32_t* meta, cudaStream_t stream);

/* ---- SURVEY.md section 8(f) row 2: modification-mode input preparation, batched -------------------------------------
 * merge_and_mask (MuseDiffusion/data/preprocess.py:30-58) + helper_filter (:73-81) + collate_batches
 * (MuseDiffusion/data/wrapper.py:90-126) for a batch of raw (src = meta tokens, trg = event tokens) pairs: every chord
 * token (195..303) of trg and the token in front of it move behind src; row = [*src', end_token, *trg'] zero padded to
 * seq_len; mask = 0 over src' + end_token, 1 elsewhere (padding included).  length[b] is the merged length; rows with
 * length > seq_len (the ones helper_filter drops) are left as pure padding.
 *   src int32 [B, Ls] + src_len [B], trg int32 [B, Lt] + trg_len [B]  ->  input_ids, input_mask int32 [B, seq_len], length [B] */
int md_merge_and_mask(const int32_t* src, const int32_t* src_len, const int32_t* trg, const int32_t* trg_len, int B, int Ls,
                      int Lt, int seq_len, int end_token, int32_t* input_ids, int32_t* input_mask, int32_t* length,
                      cudaStream_t stream);

/* ---- SURVEY.md section 8(f) row 4: sample-quality metrics on decoded note sequences, batched ------------------------
 * md_sequence_metrics: per sequence the rhythm [32] / melody [12] / harmony [12] vectors of get_vectors
 * (MuseDiffusion/metric.py:4-75; status 1 + zero vectors where the reference raises) and the token counts behind
 * Controllability_Pitch / Controllability_Velocity (:131-169).
 *   notes int32 [B, Ln] + note_len [B] (md_decode_prepare's outputs), meta int32 [B, 11]
 *   vectors f32 [B, 56] = rhythm | melody | harmony;  status int32 [B];
 *   stats int32 [B, 4] = sum and count of pitch tokens (3..130), count of velocity tokens (131..194), velocity tokens
 *   outside [meta[7] - 524, meta[8] - 524] (with the reference's 130 / 195 "unbounded" sentinels)
 * md_onnc: MSIM = product of the three Gram matrices with a zero diagonal and its row arg-max (ONNC, :89-109);
 *   vectors f32 [N, 56] -> msim f32 [N, N] (may be NULL), most_sim int32 [N]. */
int md_sequence_metrics(const int32_t* notes, const int32_t* note_len, const int32_t* meta, int B, int Ln, float* vectors,
                        int32_t* status, int32_t* stats, cudaStream_t stream);
int md_onnc(const float* vectors, int N, float* msim, int32_t* most_sim, cudaStream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* MUSEDIFF_B200_H */
