/*
 * ibm_b200.h — C ABI of libibm_b200.so, the sm_100a (B200) implementation of the
 * InferBiomechanics data-parallel hot path.
 *
 * The reference (jbejjani2022/InferBiomechanics) is 100 % Python and has no FFI layer; its hot
 * path dispatches ATen ops from the Python sites cited per entry point below (paths relative to
 * the reference root).  Each function here replaces the group of ATen launches at the cited
 * site.  INTEGRATION.md shows the ctypes binding a reference maintainer would add.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the parameter name starts with h_ (host);
 *   - the caller owns every buffer; the library allocates nothing persistent except a small
 *     per-device scratch for cross-block reductions (ibm_workspace_bytes / caller-provided);
 *   - all functions are asynchronous on `stream` (a cudaStream_t passed as void*) and re-entrant
 *     per stream; none synchronises the device;
 *   - return value: 0 on success, non-zero IBM_E_* on failure; the message is available through
 *     ibm_last_error().  There is NO CPU fallback and NO other-architecture dispatch: on a
 *     device that is not compute capability 10.x every compute entry point returns IBM_E_ARCH;
 *   - bf16 matrices are row-major with a leading dimension `ld` (elements) that must be a
 *     multiple of 8 (16-byte rows, TMA-legal); base pointers must be 16-byte aligned;
 *   - "rows30" layout: one row per (window, frame) holding the 30 output channels
 *     [CoP 6 | force 6 | torque 6 | wrench 12]  (src/models/Groundlink.py:151-156).
 */
#ifndef IBM_B200_H_
#define IBM_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define IBM_OK 0
#define IBM_E_ARG 1      /* invalid argument (shape, alignment, enum) */
#define IBM_E_ARCH 2     /* device is not sm_100 */
#define IBM_E_CUDA 3     /* CUDA runtime / driver error */
#define IBM_E_UNSUPPORTED 4

/* activation ids (src/models/FeedForwardRegressionBaseline.py:7-11; Groundlink.py:46; TransformerBaseline.py:16) */
#define IBM_ACT_NONE 0
#define IBM_ACT_RELU 1
#define IBM_ACT_SIGMOID 2
#define IBM_ACT_TANH 3
#define IBM_ACT_ELU 4
#define IBM_ACT_SILU 5

/* element types */
#define IBM_F32 0
#define IBM_BF16 1

/* ---- library ----------------------------------------------------------------------------- */
int ibm_version(void);
/* copies the calling thread's last error message; returns its length */
size_t ibm_last_error(char* buf, size_t cap);
/* 0 iff `device` is compute capability 10.x */
int ibm_device_check(int device);
/* Walk order of the big row-streaming kernels (GEMM tiles, LayerNorm rows, attention windows).  0 = ascending (default,
 * or IBM_WALK_ORDER unset); 1 = consecutive big launches alternate ascending / descending, so that a consumer starts on the
 * rows its producer wrote last (still in L2); 2 = every launch alternates, whatever its size (tests).  Results do not depend
 * on it (split-K sums are taken in a different order).  Process-wide host state: set it once, from the
 * thread that launches (the reference drives one device from one Python thread per rank, src/cli/train.py:100-102). */
int ibm_set_walk_order(int32_t mode);
/* bytes of zero-initialised device scratch the reduction kernels need (loss, layernorm bwd) */
size_t ibm_workspace_bytes(void);

/* ---- window batcher  (src/data/AddBiomechanicsDataset.py:121-139, 161-285;
 *                       src/models/FeedForwardRegressionBaseline.py:97-108) ---------------------- */

/* Candidate-window validity, Dataset.py:131-139: for candidate c of trial j (start ws),
 * valid[c] = !any(missing[ws : ws+window_size : stride]).  cand_trial/cand_start are int32[n]. */
int ibm_window_valid_mask(const uint8_t* missing, const int64_t* trial_frame_base,
                          const int32_t* cand_trial, const int32_t* cand_start, int64_t n_cand,
                          int32_t window_size, int32_t stride, uint8_t* valid, void* stream);

/* Gather F frames (stride `stride`) of each selected window from the frame store into packed
 * model inputs.  frames: fp32 [total_frames, frame_ld] whose first C columns are the model's
 * per-frame concat (FeedForward…py:97-108 order).  win_row0[i] = absolute frame index of the
 * window's first frame.  Any of out_f32 / out_bf16 may be NULL.
 *   out_f32 : [n_win, F, C] contiguous (bit-exact copy)
 *   out_bf16: element (i, f, c) at  out_bf16[(i*F + f)*bf16_frame_stride + i*bf16_win_extra + bf16_col0 + c]
 *             (round-to-nearest-even); use frame_stride=C, win_extra=ld-F*C for the FeedForward
 *             row-per-window layout, frame_stride=ld, win_extra=0 for row-per-frame layouts. */
int ibm_pack_windows(const float* frames, int64_t frame_ld, int32_t C, const int64_t* win_row0,
                     int64_t n_win, int32_t F, int32_t stride, float* out_f32, void* out_bf16,
                     int64_t bf16_frame_stride, int64_t bf16_win_extra, int64_t bf16_col0, void* stream);

/* Concatenate n_src (<= 10) fp32 tensors [n_rows, width_k] (contiguous) along the channel axis in
 * the given order (the reference's torch.concat at FeedForward…py:97-108 / Groundlink.py:122-133)
 * into packed rows; outputs addressed exactly as in ibm_pack_windows (row r = window*F + frame).
 * h_src: host array of device pointers; h_widths: host int32[n_src]. */
int ibm_pack_inputs(const void* const* h_src, const int32_t* h_widths, int32_t n_src, int64_t n_rows,
                    int32_t F, float* out_f32, void* out_bf16, int64_t bf16_frame_stride,
                    int64_t bf16_win_extra, int64_t bf16_col0, void* stream);

/* TransformerBaseline input pack (src/models/TransformerBaseline.py:108-126): the reference concatenates n_src
 * channel-major tensors (B, C_i, T) on dim 1, transposes to (B, T, C) and appends the learned temporal embedding
 * emb[t, 0:E] (expand + cat, not add).  Here: fp32 sources -> bf16 rows [B*T, ld], row b*T+t = [src_0[b,:,t] | … |
 * emb[t,:] | 0…], ld %% 8 == 0, ld >= sum C_i + E.  n_src <= 8.  Bit-exact RNE bf16 of the fp32 values. */
int ibm_pack_channel_major(const void* const* srcs, const int32_t* channels, int32_t n_src, int64_t B, int32_t T,
                           const float* emb, int32_t E, void* out_bf16, int64_t ld, void* stream);

/* Pre-packed analysis stream: rows converted once on the host to frame-major bf16 [n_rows = B*T, ld_src] (C channels per frame)
 * -> the TransformerBaseline's input rows [n_rows, ld] = [C channels | E temporal-embedding columns of frame r % T | zeros],
 * bit-identical to ibm_pack_channel_major on the fp32 (B, C, T) tensors (TransformerBaseline.py:108-126); v_out (may be NULL):
 * bf16 [n_rows, 8] <- columns [v_col0, v_col0+3) | zeros (the CoM accelerations blended by SimpleAttention, …:135-137). */
int ibm_expand_rows_bf16(const void* src_bf16, int64_t ld_src, int32_t C, int64_t n_rows, int32_t T, const float* emb,
                         int32_t E, void* out_bf16, int64_t ld, void* v_out_bf16, int32_t v_col0, void* stream);

/* Label rows (Dataset.py:216-261): raw first-pass per-frame [cop 3nb | force 3nb | torque 3nb |
 * wrench 6nb] in the SUBJECT's body order → rows30 in the DATASET's body order, force/torque/
 * wrench divided by the subject mass (IEEE fp32 division), absent bodies → 0.
 * contact_idx: int32 [n_win, nb]; mass: fp32 [n_win].  last_frame_only!=0 keeps only frame F-1. */
int ibm_pack_labels(const float* raw, int64_t raw_ld, int32_t nb, const int64_t* win_row0,
                    const int32_t* contact_idx, const float* mass, int64_t n_win, int32_t F,
                    int32_t stride, int32_t last_frame_only, float* out_rows, int64_t out_ld, void* stream);

/* ---- regression loss  (src/loss/RegressionLossEvaluator.py:160-221 step 1, 230-263 step 2.2) ----- */

/* Quantity order everywhere: 0 CoP, 1 force, 2 torque, 3 wrench (6,6,6,12 channels).
 * h_out / h_lab: host arrays of 4 device pointers (fp32); h_out_strides / h_lab_strides: host
 * int64[8] = {stride_b, stride_f} per quantity in elements (channel stride is 1).
 * h_weights: host fp32[30] = multiplicity of each component in the args.predict_* lists
 * (…py:217-220; a repeated index counts twice, an absent one 0).
 * result: fp32[40] = loss, then the 30 per-component means in quantity order cop[6], force[6],
 * moment[6], wrench[12], then reports{force, moment, cop, wrench_moment, wrench, com_acc}
 * (last frame only, …py:119-158), 3 pad.
 * workspace: ibm_workspace_bytes() of zeroed device memory (left zeroed on return). */
int ibm_regression_loss_fwd(const void* const* h_out, const int64_t* h_out_strides,
                            const void* const* h_lab, const int64_t* h_lab_strides,
                            int64_t B, int64_t F, const float* h_weights, float threshold,
                            float* result, void* workspace, void* stream);

/* d loss / d outputs = upstream * 2 w_c m^2 (o-l) / (B*F)   (SURVEY §9.1).
 * upstream: device fp32 scalar (NULL ⇒ 1).  h_grad: host array of 4 device pointers of
 * grad_dtype (IBM_F32 | IBM_BF16) with h_grad_strides like h_out_strides. */
int ibm_regression_loss_bwd(const void* const* h_out, const int64_t* h_out_strides,
                            const void* const* h_lab, const int64_t* h_lab_strides,
                            int64_t B, int64_t F, const float* h_weights, float threshold,
                            const float* upstream, void* const* h_grad, const int64_t* h_grad_strides,
                            int32_t grad_dtype, void* stream);

/* ---- the loss evaluator's four static helpers with their general contract -------------------------
 * (src/loss/RegressionLossEvaluator.py:73-158; exercised by test/loss/test_RegressionLossEvaluator.py)
 * All tensors are fp32 (B, F, C) views with unit channel stride; sb / sf = batch / frame strides in
 * elements.  workspace: ibm_workspace_bytes() of zeroed device memory (left zeroed on return).
 * IBM_E_ARG carries the reference's ValueError text (empty tensor, C % 3, C % vec_size, C != 6). */

/* get_squared_diff_mean_vector (…py:73-83): result[c] = mean over (b, f) of (out-lab)^2, any C. */
int ibm_sqdiff_mean_vector(const float* out_t, int64_t o_sb, int64_t o_sf, const float* lab_t, int64_t l_sb,
                           int64_t l_sf, int64_t B, int64_t F, int32_t C, float* result, void* workspace,
                           void* stream);
/* its autograd backward: grad_out[b,f,c] = 2 upstream[c] (out-lab) / (B F) (contiguous (B,F,C)); grad_lab is
 * the negative.  Either may be NULL. */
int ibm_sqdiff_mean_vector_bwd(const float* out_t, int64_t o_sb, int64_t o_sf, const float* lab_t, int64_t l_sb,
                               int64_t l_sf, int64_t B, int64_t F, int32_t C, const float* upstream,
                               float* grad_out, float* grad_lab, void* stream);
/* get_mask_by_threes (…py:85-108): mask[b,f,3g:3g+3] = (||x[b,f,3g:3g+3]||_2 > threshold) ? 1 : 0, strict >,
 * bit-exact; mask is contiguous fp32 (B,F,C); C % 3 == 0. */
int ibm_mask_by_threes(const float* x, int64_t sb, int64_t sf, int64_t B, int64_t F, int32_t C, float threshold,
                       float* mask, void* stream);
/* get_mean_norm_error (…py:119-141): result[0] = mean over (b, g) of ||(out-lab)[b, F-1, g v:(g+1) v]||_2 — last
 * frame only; C % vec_size == 0.  fold_halves = 1 is get_com_acc_error (…py:143-158): C == 6, the two 3-vectors of
 * each tensor are summed first. */
int ibm_mean_norm_error(const float* out_t, int64_t o_sb, int64_t o_sf, const float* lab_t, int64_t l_sb, int64_t l_sf,
                        int64_t B, int64_t F, int32_t C, int32_t vec_size, int32_t fold_halves, float* result,
                        void* workspace, void* stream);

/* ---- DDPM (builder-owned spec, DESIGN.md D-1; NOT in the reference) --------------------------- */

/* x_t = sqrt_abar[t_b] x0 + sqrt_1m_abar[t_b] eps.  x0/eps/xt_f32: fp32 [B, per_win] contiguous
 * (per_win = F*30).  If eps == NULL, eps is drawn on-device from Philox4x32-10(seed, offset) and
 * (if eps_out != NULL) written there.  xt_bf16 (optional): rows30 scattered into a bf16 matrix:
 * element (m, c) at xt_bf16[m*bf16_ld + c], m = b*F + f. */
int ibm_q_sample(const float* x0, const float* eps, const int32_t* t, const float* sqrt_abar,
                 const float* sqrt_1m_abar, int64_t B, int64_t per_win, float* xt_f32,
                 void* xt_bf16, int64_t bf16_ld, uint64_t seed, uint64_t offset, float* eps_out,
                 void* stream);

/* x_{t-1} = c1[t] x0_hat + c2[t] x_t + [t>0] sigma[t] z  for one shared timestep t (read from
 * device int32 *t_dev so the sampling loop can live in a CUDA graph).  x0_hat: fp32 rows with
 * leading dim x0_ld (30 used); x_t / z / x_prev: fp32 [M,30] contiguous; z == NULL ⇒ Philox.
 * xprev_bf16 optional as in ibm_q_sample.  If t_next_dev != NULL it receives t-1. */
int ibm_ddpm_posterior_step(const float* x0_hat, int64_t x0_ld, const float* x_t, const float* z,
                            const int32_t* t_dev, const float* coef_x0, const float* coef_xt,
                            const float* sigma, int64_t M, float* x_prev, void* xprev_bf16,
                            int64_t bf16_ld, uint64_t seed, uint64_t offset, int32_t* t_next_dev,
                            void* stream);

/* One step of a respaced sampler (DDIM, DESIGN.md D-1) with the arguments and semantics of
 * ibm_ddpm_posterior_step: x_p = coef_x0[t] x0_hat + coef_xt[t] x_t + [t>0] sigma[t] z, Philox counter
 * offset + t.  The tables hold the coefficients of the step from t to its successor p, and
 * t_succ (device int32 [T]) names p: t_next_dev, if not NULL, receives t_succ[t] instead of t-1. */
int ibm_ddpm_respaced_step(const float* x0_hat, int64_t x0_ld, const float* x_t, const float* z,
                           const int32_t* t_dev, const float* coef_x0, const float* coef_xt,
                           const float* sigma, int64_t M, float* x_prev, void* xprev_bf16,
                           int64_t bf16_ld, uint64_t seed, uint64_t offset, int32_t* t_next_dev,
                           const int32_t* t_succ, void* stream);

/* Classifier-free guidance (DESIGN.md D-1).  One step of ibm_ddpm_posterior_step (t_succ == NULL) or
 * ibm_ddpm_respaced_step (t_succ != NULL) on a guided prediction: x0_hat holds 2M rows (leading dim
 * x0_ld), rows 0..M-1 conditional (c) and rows M..2M-1 unconditional (u), combined per element in fp32 as
 * fmaf(guidance_scale, c - u, u) before the unchanged update, [t>0] noise gate and Philox counter
 * offset + t.  x_t / z / x_prev: fp32 [M,30]; xprev_bf16 (optional) receives the bf16 rows twice, at
 * rows m and M + m, so both halves of the next forward see the same x_t.  guidance_scale: finite, >= 0. */
int ibm_ddpm_guided_step(const float* x0_hat, int64_t x0_ld, const float* x_t, const float* z,
                         const int32_t* t_dev, const float* coef_x0, const float* coef_xt,
                         const float* sigma, int64_t M, float* x_prev, void* xprev_bf16,
                         int64_t bf16_ld, uint64_t seed, uint64_t offset, int32_t* t_next_dev,
                         const int32_t* t_succ, float guidance_scale, void* stream);

/* Builder-owned (DESIGN.md D-1; NOT in the reference): inpainting.  One step of ibm_ddpm_guided_step (guided != 0) or of
 * the unguided posterior / respaced step (guided == 0; t_succ selects as there, guidance_scale is checked and unused) in
 * which the known entries of the prediction are held fixed: after the guided combination, and before the unchanged update,
 * [t>0] noise gate and Philox counter offset + t,
 *   x0_hat[m, c] = known[m, c]  where bit c of known_mask[m] is set,  else the prediction.
 * A select, not a blend: an entry of `known` whose bit is clear is never read into the result (it may hold NaN).
 * known: fp32 [M, 30] contiguous, 8-byte aligned.  known_mask: int32 [M], one word per row, bits 0..29 = channels,
 * bits 30-31 ignored.  Both are required; everything ibm_ddpm_guided_step refuses is refused too. */
int ibm_ddpm_inpaint_step(const float* x0_hat, int64_t x0_ld, const float* x_t, const float* z,
                          const int32_t* t_dev, const float* coef_x0, const float* coef_xt,
                          const float* sigma, int64_t M, float* x_prev, void* xprev_bf16,
                          int64_t bf16_ld, uint64_t seed, uint64_t offset, int32_t* t_next_dev,
                          const int32_t* t_succ, float guidance_scale, int32_t guided, const float* known,
                          const int32_t* known_mask, void* stream);

/* Per-window condition dropout for classifier-free guidance training.  xc: bf16 [B*F, ld] (window b
 * owns rows b*F .. b*F+F-1).  Window b is dropped iff word 0 of Philox4x32-10 draw b at (seed, offset)
 * is below uint32(p * 2^32) (the keep rule of the dropout kernels); p >= 1 drops every window without
 * drawing.  A dropped window gets +0 in columns col0 .. col0+ncols-1 of its F rows; no other byte is
 * written.  keep_out (optional): uint8 [B], 1 = kept, 0 = dropped.  Requires 0 < p. */
int ibm_cond_dropout(void* xc_bf16, int64_t ld, int64_t B, int32_t F, int32_t col0, int32_t ncols, float p,
                     uint64_t seed, uint64_t offset, uint8_t* keep_out, void* stream);

/* Builder-owned (DESIGN.md §3; NOT in the reference): probabilistic score of K sampled trajectories per window.
 * draws: fp32 [K, B*F, 30] draw-major (draw k of window b, frame f at row k*B*F + b*F + f), the fp32 state
 * GaussianDiffusion.sample returns for B*K windows whose conditions are K copies of the same B.  labels: fp32 [B, Fo, 30]
 * (rows30); Fo = F scores every frame, Fo = 1 (last_frame) scores frame F-1 of each draw.  For each scored element with
 * draws x_1..x_K and label y:
 *   m    = (1/K) sum_k x_k                      (fp64 sum; written to mean_out fp32 [B, Fo, 30] as rounded)
 *   s2   = 1/(K-1) sum_k (x_k - m)^2            (two-pass, from m)
 *   pair = 1/(K(K-1)) sum_{i!=j} |x_i - x_j|    (mean pairwise distance: a per-component MDM MultiModality)
 *   crps = (1/K) sum_k |x_k - y| - pair/2       (the fair CRPS, Ferro 2014: unbiased at every K)
 *   se   = (m - y)^2
 * CoP channels 0-2 (3-5) are scored only on rows whose label force triple 6-8 (9-11) passes the contact test of
 * ibm_regression_loss_fwd at `threshold` (||f|| > threshold, bit for bit the same predicate); every other channel is scored
 * on every row.  mean_out is written for every element.
 * acc: fp64 [5, 30], caller-owned, row q channel c: += the batch's sum over scored elements of channel c of
 *   q = 0 crps, 1 s2, 2 se, 3 pair, 4 the element count,
 * so successive batches accumulate on the device.  Per-block partials and a last-arriving-block reduction in a fixed order:
 * the same inputs on the same device give bit-identical accumulators.  Workspace, caller-owned: partials = 1024 * 150
 * doubles, counter = one uint32 that is zero before the first call (the kernel resets it).  2 <= K <= 64: the kernel holds
 * the K draws of an element in registers.  Buffers contiguous, fp32 ones 4-byte and fp64 ones 8-byte aligned.  No allocation
 * or host synchronisation: the call can be captured in a CUDA graph. */
int ibm_ensemble_score(const float* draws, int32_t K, int64_t B, int32_t F, const float* labels, int32_t Fo, float threshold,
                       float* mean_out, double* acc, double* partials, uint32_t* counter, void* stream);

/* sinusoidal timestep embedding, bf16 [B, dim] (ld = dim): [sin(t w_k) | cos(t w_k)],
 * w_k = 10000^(-k/(dim/2)).  t: int32[B], or if t_is_scalar a single device int32 broadcast. */
int ibm_timestep_embed(const int32_t* t, int32_t t_is_scalar, int64_t B, int32_t dim, void* out_bf16,
                       void* stream);

/* h[m,:] += temb[m / F, :] + pos[m % F, :]   (bf16 in place; temb bf16 [B,d]; pos fp32 [F,d]).
 * t_row_dev != NULL (reverse sampling: every window is at the same timestep): temb is a table with one row per
 * timestep and row t_row_dev[0] (a device int32) is added to every window, so the time MLP is evaluated once per
 * model, not once per denoise step. */
int ibm_add_time_pos(void* h_bf16, int64_t ld, const void* temb_bf16, int64_t temb_ld,
                     const float* pos, int64_t M, int32_t F, int32_t d, const int32_t* t_row_dev, void* stream);
/* backward of the above in ONE pass over dh: dtemb[b,:] = sum_f dh[b,f,:] (bf16 out); dpos[f,:] += sum_b dh[b,f,:] (fp32
 * atomic); dbias (may be NULL): fp32 [d] += sum_{b,f} dh[b,f,:] — the bias gradient of the Linear that produced h (the
 * denoiser's in-projection), which would otherwise be a second full read of dh. */
int ibm_add_time_pos_bwd(const void* dh_bf16, int64_t ld, void* dtemb_bf16, int64_t temb_ld,
                         float* dpos, int64_t M, int32_t F, int32_t d, float* dbias, void* stream);

/* ---- dense layers  (nn.Linear sites: FeedForward…py:73,113; Groundlink.py:51-62;
 *                     TransformerBaseline.py:12-18,91; nn.Conv1d: Groundlink.py:41) --------------- */

/* D[M,N] (+)= epilogue( A · B^T )  on tcgen05 tensor cores, bf16 operands, fp32 accumulation.
 *   A: bf16, logical [M,K]. a_mn_major==0: stored row-major [M,K] (ld=lda).
 *                           a_mn_major==1: stored row-major [K,M] (ld=lda)  (i.e. A^T in memory).
 *   B: bf16, logical [N,K]. b_mn_major likewise ([N,K] vs [K,N] in memory).
 *   bias: fp32[N], 16-byte aligned, or NULL.  act: IBM_ACT_* applied to (acc + bias).
 *   aux: bf16 [M,N] (ld=ldaux) or NULL; aux_mode 1: out = act(acc+bias) + aux   (residual; act none/relu/elu)
 *                                        aux_mode 2: out = (acc+bias) * act'(aux) (aux = saved
 *                                        activation OUTPUT; dgrad through none/relu/sigmoid/tanh/elu)
 *   Other act with aux, and any act with mask_mode 2, are rejected (IBM_E_ARG).
 *   out: out_dtype IBM_BF16 | IBM_F32, row-major [M,N] (ld=ldd).
 *   accumulate!=0 (requires IBM_F32 out, no act/aux): D += A·B^T via TMA reduce-add; the K range is
 *   split over `split_k` CTAs (weight gradients: K = tokens).  split_k<=0 ⇒ chosen by the library.
 *   taps>1: A rows are shifted by tap index: K is taps*K_tap, k-block kb reads A rows
 *   m + (kb / kb_per_tap) (implicit-GEMM temporal convolution, Groundlink.py:41).  B holds taps blocks of
 *   round_up(K_tap, 64) k: tap j's weights start at k = j * round_up(K_tap, 64) (B is [N, taps*round_up(K_tap, 64)],
 *   or its transpose when MN-major).
 *   colsum_out: NULL, or fp32[N] that the column sums of the bf16 output (rows < M, as rounded) are
 *   ADDED to by the epilogue: when D is the gradient w.r.t. a layer's pre-activation this is that
 *   layer's bias gradient (nn.Linear bias, TransformerBaseline.py:15) without another pass over D.
 *   mask / ldmask / mask_mode: sign bitmask [M][ldmask bytes] (bit c&7 of byte c>>3 <-> column c; bf16 output,
 *   N %% 64 == 0, no aux).  mask_mode 1 (forward of Linear+ReLU, TransformerBaseline.py:15-16): bit = (D > 0) is
 *   written next to D.  mask_mode 2 (its dgrad): D = (acc + bias) where the bit is set, 0 elsewhere — the ReLU
 *   derivative from 1 bit per element instead of re-reading the saved activation (aux_mode 2).  0: unused. */
int ibm_gemm_bf16(const void* A, int64_t lda, int32_t a_mn_major, const void* B, int64_t ldb,
                  int32_t b_mn_major, int64_t M, int64_t N, int64_t K, const float* bias, int32_t act,
                  const void* aux, int64_t ldaux, int32_t aux_mode, void* D, int64_t ldd,
                  int32_t out_dtype, int32_t accumulate, int32_t split_k, int32_t taps, float* colsum_out, void* mask,
                  int64_t ldmask, int32_t mask_mode, void* stream);

/* out[n] (+)= sum_m X[m,n]   (bias gradients; X bf16 [M,N] ld; out fp32; accumulate via atomics) */
int ibm_colsum_bf16(const void* X, int64_t ld, int64_t M, int64_t N, float* out, void* stream);

/* y = act(x) elementwise bf16→bf16 and its backward dx = dy*act'(x) (x = pre-activation) */
int ibm_act_fwd(const void* x, void* y, int64_t n, int32_t act, void* stream);
int ibm_act_bwd(const void* dy, const void* x, void* dx, int64_t n, int32_t act, void* stream);

/* fp32 → bf16 (RNE) flat cast; n elements */
int ibm_cast_f32_bf16(const float* src, void* dst, int64_t n, void* stream);
/* bf16 → fp32 flat cast */
int ibm_cast_bf16_f32(const void* src, float* dst, int64_t n, void* stream);
/* strided 2-D cast fp32 [rows, cols] (ld_src) → bf16 (ld_dst), zero-filling cols..ld_dst */
int ibm_cast_pad_f32_bf16(const float* src, int64_t ld_src, void* dst, int64_t ld_dst, int64_t rows,
                          int64_t cols, void* stream);
/* Conv1d weight (Cout,Cin,Kt) fp32 → bf16 GEMM layout [Cout, Kt*cin_pad], (tap, ci) order */
int ibm_conv_weight_to_gemm(const float* w, int32_t cout, int32_t cin, int32_t kt, int32_t cin_pad,
                            void* dst_bf16, void* stream);
/* inverse for gradients: dW_gemm fp32 [Cout, Kt*cin_pad] → (Cout,Cin,Kt) fp32 (+= if accumulate) */
int ibm_conv_wgrad_from_gemm(const float* g, int32_t cout, int32_t cin, int32_t kt, int32_t cin_pad,
                             float* dw, int32_t accumulate, void* stream);

/* Temporal replicate padding for the implicit-GEMM convolution (Groundlink.py:41, padding_mode="replicate").
 * Padded row layout: window b owns rows [b*Tp, (b+1)*Tp), Tp = T + 2*pad, frame t at row b*Tp + pad + t.
 * replicate: pad rows <- first / last frame row.  fold (its adjoint): edge frame rows += pad rows, pad rows <- 0
 * (T == 1: the one frame row gains both sides' pad rows).  T > 0, pad >= 0; pad == 0 (kernel size 1) is a no-op. */
int ibm_replicate_pad_rows(void* X_bf16, int64_t ld, int64_t n_win, int32_t T, int32_t pad, int32_t cols, void* stream);
int ibm_fold_pad_rows(void* G_bf16, int64_t ld, int64_t n_win, int32_t T, int32_t pad, int32_t cols, void* stream);
/* Inverted dropout (nn.Dropout, Groundlink.py:53,59): y = x * keep/(1-p), keep from Philox4x32-10(seed, offset);
 * the backward pass calls it on dy with the same (seed, offset).  n % 4 == 0. */
int ibm_dropout_bf16(const void* x, void* y, int64_t n, float p, uint64_t seed, uint64_t offset, void* stream);
/* Same mask generator with the Philox offset = offset + step_mul * *step_dev, the step read from device memory at execution
 * time (graph-replayed training steps draw a fresh mask per replay; forward and backward of one step see the same value). */
int ibm_dropout_bf16_dev(const void* x, void* y, int64_t n, float p, uint64_t seed, uint64_t offset,
                         const int64_t* step_dev, int64_t step_mul, void* stream);
/* Conv1d weight (Cout,Cin,Kt) fp32 -> bf16 dgrad layout [Cin, Kt*cout_pad]: B[ci, j*cout_pad+co] = W[co,ci,Kt-1-j] */
int ibm_conv_weight_to_dgrad(const float* w, int32_t cout, int32_t cin, int32_t kt, int32_t cout_pad,
                             void* dst_bf16, void* stream);

/* ---- BatchNorm1d on the layer input  (src/models/FeedForwardRegressionBaseline.py:71-72; nn.BatchNorm1d defaults
 *      eps=1e-5, momentum=0.1, affine, track_running_stats) ---- */

/* floats of caller-owned scratch the two BatchNorm entry points need for C features */
size_t ibm_batchnorm_workspace_floats(int32_t C);
/* y = (x - mean) / sqrt(var + eps) * gamma + beta per column.  x,y bf16 [M, ld] (ld %% 8 == 0; columns C..ld of y are
 * written 0); gamma/beta fp32[C].  training != 0: mean / biased variance of THIS batch (two-pass per row chunk, chunks
 * merged with Chan's update), saved as save_mean / save_rstd fp32[C] for the backward pass; running_mean / running_var
 * (fp32[C], may be NULL) are updated in place with `momentum` and the UNBIASED batch variance; M == 1 is an argument
 * error like torch's ValueError.  training == 0: normalises with running_mean / running_var; save_* and workspace unused. */
int ibm_batchnorm_fwd(const void* x, int64_t ldx, void* y, int64_t ldy, int64_t M, int32_t C, const float* gamma,
                      const float* beta, float* running_mean, float* running_var, float* save_mean, float* save_rstd,
                      int32_t training, float momentum, float eps, float* workspace, void* stream);
/* Backward of the above.  dgamma[c] += sum_m dy*xhat, dbeta[c] += sum_m dy (either may be NULL);
 * dx = gamma*rstd*(dy - mean_m(dy) - xhat*mean_m(dy*xhat)) in training mode, gamma*rstd*dy in eval mode (dx may be NULL
 * when only the parameter gradients are wanted, may alias dy).  (mean, rstd_or_var) = (save_mean, save_rstd) when
 * training, (running_mean, running_var) otherwise.  act_out != NULL: dx is additionally multiplied by act'(.) expressed
 * through the saved activation OUTPUT act_out (the activation that produced x's layer input; relu/sigmoid/tanh/elu).
 * dx_colsum (fp32[C], may be NULL): += column sums of dx taken in fp32 before the bf16 rounding — the bias gradient of
 * the Linear that feeds this BatchNorm (a sum of cancelling terms in training mode). */
int ibm_batchnorm_bwd(const void* dy, int64_t lddy, const void* x, int64_t ldx, void* dx, int64_t lddx, int64_t M,
                      int32_t C, const float* gamma, const float* mean, const float* rstd_or_var, int32_t training,
                      float eps, const void* act_out, int64_t ldact, int32_t act, float* dgamma, float* dbeta,
                      float* dx_colsum, float* workspace, void* stream);

/* ---- residual + LayerNorm  (src/models/TransformerBaseline.py:31,36; nn.LayerNorm eps=1e-5) ---- */

/* y = LN(s) * gamma + beta over the first d columns of each row (columns d..ld are written 0).
 * s,y bf16 [M, ld]; gamma/beta fp32[d]; mean/rstd fp32[M] saved for backward (may be NULL). */
int ibm_layernorm_fwd(const void* s, void* y, int64_t ld, const float* gamma, const float* beta,
                      int64_t M, int32_t d, float eps, float* mean, float* rstd, void* stream);
/* ds = LN'(dy); dgamma += sum dy*xhat; dbeta += sum dy; if dcolsum != NULL: dcolsum += colsum(ds)
 * (bias gradient of the linear layer that produced s).  fp32 atomics into dgamma/dbeta/dcolsum. */
int ibm_layernorm_bwd(const void* dy, const void* s, int64_t ld, const float* gamma,
                      const float* mean, const float* rstd, int64_t M, int32_t d, void* ds,
                      float* dgamma, float* dbeta, float* dcolsum, void* stream);

/* ---- attention  (nn.MultiheadAttention, src/models/TransformerBaseline.py:12-13,29) ----------- */

/* Whole-sequence softmax attention per (window, head): o = softmax(scale * q k^T) v.
 * q,k,v,o: bf16 matrices with one row per (window, frame) (n_win*T rows); head h occupies columns
 * [h*hd_qk, (h+1)*hd_qk) of q and k and [h*hd_v, (h+1)*hd_v) of v and o.  For a fused QKV
 * projection pass q = qkv, k = qkv + kv_off, v = qkv + 2*kv_off with ldq = ldk = ldv.
 * Supported (hd_qk, hd_v): (64,64) (48,48) (32,32) and (112,8) — the latter is SimpleAttention
 * (TransformerBaseline.py:51-70: scale = 1, d = 108 padded to 112, value dim 3 padded to 8).
 * T <= 256 (whole K and V of a head live in shared memory). */
int ibm_attention_fwd(const void* q, int64_t ldq, const void* k, int64_t ldk, const void* v, int64_t ldv,
                      void* o, int64_t ldo, int64_t n_win, int32_t T, int32_t H, int32_t hd_qk,
                      int32_t hd_v, float scale, void* stream);
/* dqkv (same layout as qkv: q | k | v blocks kv_off columns apart) from d_o; probabilities are
 * recomputed on chip.  T <= 64, head_dim in {32,48,64}.  dbias_qkv (may be NULL): fp32
 * [2*kv_off + H*head_dim] vector that the column sums of dqkv are ADDED to — the gradient of
 * nn.MultiheadAttention.in_proj_bias (TransformerBaseline.py:12) without a second pass over dqkv. */
int ibm_attention_bwd(const void* qkv, int64_t ld_qkv, int64_t kv_off, const void* d_o, int64_t ld_o,
                      void* dqkv, int64_t n_win, int32_t T, int32_t H, int32_t head_dim, float scale,
                      float* dbias_qkv, void* stream);

/* Backward of the same attention for whole windows of up to 256 frames (the reference's own TransformerBaseline shapes:
 * 3 heads x 36 -> 48 padded at T = window_size, TransformerBaseline.py:12-13,29; and SimpleAttention, …:51-70, with
 * (hd_qk, hd_v) = (112, 8), dv = NULL because its values are a model INPUT).  q,k,v,o,d_o as in ibm_attention_fwd
 * (o = the forward output); dq,dk,dv: bf16 outputs with their own leading dimensions (head h at columns h*hd).
 * Probabilities are recomputed on chip.  dbias_q/k/v (each may be NULL): fp32 [H*hd] vectors the column sums of
 * dq/dk/dv are ADDED to (in_proj_bias / query_linear.bias / key_linear.bias gradients).
 * Supported: (64,64) (48,48) (32,32) with dv, (112,8) without. */
int ibm_attention_bwd_long(const void* q, int64_t ldq, const void* k, int64_t ldk, const void* v, int64_t ldv,
                           const void* o, int64_t ldo, const void* d_o, int64_t ld_do, void* dq, int64_t lddq,
                           void* dk, int64_t lddk, void* dv, int64_t lddv, int64_t n_win, int32_t T, int32_t H,
                           int32_t hd_qk, int32_t hd_v, float scale, float* dbias_q, float* dbias_k, float* dbias_v,
                           void* stream);

/* ---- optimizers  (src/cli/train.py:183-197, 284; torch.optim defaults) ------------------------ */

/* One fused step over a flat fp32 parameter arena: reads grad (scaled by grad_scale, e.g.
 * 1/world_size after an allreduce-sum), updates param and optimizer state in place, and writes
 * the bf16 shadow copy used by the GEMMs.  kind: 0 rmsprop(alpha .99, eps 1e-8), 1 adam(.9,.999,
 * 1e-8), 2 sgd, 3 adagrad(eps 1e-10), 4 adadelta(rho .9, eps 1e-6), 5 adamax(.9,.999,1e-8).
 * state0/state1: fp32 arenas (unused ones may be NULL).  step = 1-based step count. */
int ibm_optimizer_step(int32_t kind, float* param, const float* grad, float* state0, float* state1,
                       void* param_bf16, int64_t n, float lr, float grad_scale, int64_t step,
                       void* stream);
/* Same step with the 1-based step count read from DEVICE memory (int64[1]) at execution time: a captured CUDA graph of the
 * training step can be replayed although Adam / Adamax bias corrections change every step. */
int ibm_optimizer_step_dev(int32_t kind, float* param, const float* grad, float* state0, float* state1,
                           void* param_bf16, int64_t n, float lr, float grad_scale, const int64_t* step_dev,
                           void* stream);
/* Builder-owned (DESIGN.md §0; NOT in the reference): the same step, and in the same pass an exponential moving average of the
 * updated parameters in the fp32 arena `ema` (same offsets as param, 16-byte aligned):
 *   d_n = min(ema_decay, (1 + n) / (10 + n))   (double; n = the 1-based step count)
 *   ema <- ema + (float)(1 - d_n) * (param - ema)
 * 0 < ema_decay < 1.  n = step, or *step_dev when step_dev != NULL (graph-replayed steps). */
int ibm_optimizer_step_ema(int32_t kind, float* param, const float* grad, float* state0, float* state1,
                           void* param_bf16, float* ema, int64_t n, float lr, float grad_scale, float ema_decay,
                           int64_t step, const int64_t* step_dev, void* stream);
/* Builder-owned (DESIGN.md §0; NOT in the reference): global gradient norm and clip coefficient of
 * torch.nn.utils.clip_grad_norm_(params, max_norm) over the flat fp32 gradient arena (16-byte aligned):
 *   total = grad_scale * ||grad||_2   (fp64 per thread and per block, deterministic last-block reduction, rounded to fp32)
 *   coef  = min(1, max_norm / (total + 1e-6))   (fp32, as torch; a NaN total gives a NaN coefficient)
 * out = {total, coef} (device float[2]).  The norm covers the whole arena, so the alignment padding between parameters
 * must be zero, which it is when the arena is cleared as a whole before backward and nothing writes the padding.
 * Workspace, caller-owned: partials = 1024 doubles, counter = one uint32 that is zero before the first call (the kernel
 * resets it).  record (nullable, device double[3]): += {total, 1, coef < 1 ? 1 : 0}, a running sum for reports.
 * No allocation, host synchronisation or host read: the call can be captured in a CUDA graph.  Two calls on the same
 * arena and device give bit-identical outputs; max_norm > 0. */
int ibm_grad_clip_coef(const float* grad, int64_t n, float grad_scale, float max_norm, float* out, double* partials,
                       uint32_t* counter, double* record, void* stream);
/* Builder-owned (DESIGN.md §0; NOT in the reference): ibm_optimizer_step_ema with `ema` nullable, a clip coefficient and a
 * learning-rate schedule, both applied on the device so that a captured step replays with the values of its own step:
 *   gradient = (grad * grad_scale) * clip[1]   (clip: the float[2] of ibm_grad_clip_coef, or NULL for no clipping)
 *   lr_n     = (float)((double)lr * lambda(n)), n = the 1-based step (step, or *step_dev when step_dev != NULL), with
 *     lambda(n) = n / W                                    for W > 0 and n <= W   (linear warm-up, W = warmup_steps)
 *               = 1                                        after the warm-up, sched 0 (constant)
 *               = r + (1 - r) (1 + cos(pi p)) / 2          after the warm-up, sched 1 (cosine), r = lr_min / lr,
 *                 p = clamp((n - W) / (S - W), 0, 1), S = total_steps
 * lr_n is the rate torch.optim.lr_scheduler.LambdaLR(opt, lambda s: lambda(s + 1)) hands to the optimizer's n-th step().
 * warmup_steps >= 0; sched 1 needs total_steps > warmup_steps; 0 <= lr_min <= lr.  With clip[1] == 1 and lambda == 1 the
 * update is bit-identical to ibm_optimizer_step_dev / _ema (both factors multiply by exactly 1). */
int ibm_optimizer_step_sched(int32_t kind, float* param, const float* grad, float* state0, float* state1,
                             void* param_bf16, float* ema, int64_t n, float lr, float grad_scale, float ema_decay,
                             int64_t step, const int64_t* step_dev, const float* clip, int32_t sched,
                             int64_t warmup_steps, int64_t total_steps, float lr_min, void* stream);
/* *counter_dev += inc (one thread): the device-resident step counter of graph-replayed training steps. */
int ibm_counter_add(int64_t* counter_dev, int64_t inc, void* stream);

/* ---- diagnostics ---------------------------------------------------------------------------- */

/* How many thread-block clusters of `cluster_size` CTAs of the 256 x 256 GEMM kernel can be resident at once
 * (cudaOccupancyMaxActiveClusters).  On B200: 74 pairs, 33 quads, 15 octets — why the GEMM uses CTA pairs and
 * two-tile work items rather than larger multicast clusters (DESIGN.md section 6).  Returns -1 on error. */
int ibm_debug_gemm_max_clusters(int32_t cluster_size);

#ifdef __cplusplus
}
#endif
#endif /* IBM_B200_H_ */
