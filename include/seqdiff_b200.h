/*
 * seqdiff_b200.h -- C ABI of libseqdiff_b200.so: the B200 (sm_100a) implementation of ONE hot path of
 * LabJunBMI/E3-invaraint-diffusion-model: the sequence_model denoiser forward and the discrete
 * BLOSUM-transition reverse-diffusion step -- plus, widening along SURVEY.md section 8(f), the output decode, the loss
 * reductions and the structure_model angle denoiser with its Gaussian reverse step on the same kernels.
 *
 * The reference is pure Python/PyTorch and has no FFI layer (SURVEY.md section 8b); the boundary a
 * maintainer binds is therefore "one entry point per reference function on the path".  Each entry
 * point below names the reference interface it replaces (paths relative to the reference root).
 * INTEGRATION.md shows the ctypes stub that goes into the reference's model.py / sample.py.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the parameter name ends in `_host`;
 *   - all tensors are dense, row-major, caller-owned; nothing is allocated for or freed on behalf of
 *     the caller; a model handle owns its packed weights and its workspace;
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream); calls are
 *     asynchronous on that stream and re-entrant per handle+stream pair;
 *   - return value 0 = SEQDIFF_OK, otherwise an error code; seqdiff_last_error() returns the
 *     thread-local message.  There is NO CPU fallback: without a CUDA device every compute entry
 *     point returns SEQDIFF_ERR_CUDA.
 */
#ifndef SEQDIFF_B200_H_
#define SEQDIFF_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define SEQDIFF_API __attribute__((visibility("default")))
#else
#define SEQDIFF_API
#endif

#define SEQDIFF_ABI_VERSION 1

#define SEQDIFF_OK 0
#define SEQDIFF_ERR_INVALID 1   /* bad argument / unsupported shape            */
#define SEQDIFF_ERR_CUDA 2      /* CUDA runtime / driver error                 */
#define SEQDIFF_ERR_STATE 3     /* handle not finalised, unknown tensor name   */

/* precision modes.  In every 16-bit mode the GEMM/attention OPERANDS are 16-bit while accumulators, the
 * residual stream, LayerNorm, softmax, biases and logits stay fp32. */
#define SEQDIFF_FP32 0       /* fp32 everything, SIMT GEMMs                      (parity gate 1e-5) */
#define SEQDIFF_BF16 1       /* bf16 activations x bf16 weights, tcgen05 GEMMs   (the named config) */
#define SEQDIFF_FP16 2       /* fp16 activations x fp16 weights, same kernels, 8x finer mantissa    */
/* (A and B of one tcgen05.mma.kind::f16 must share a format: a bf16 x fp16 mix traps as an illegal
 * instruction on B200, measured in round 1, so there is no mixed mode.) */

#define SEQDIFF_NUM_CLASSES 20
#define SEQDIFF_ANGLE_FEATS 8

typedef struct seqdiff_model seqdiff_model_t;

/* The BertConfig fields the path consumes: sequence_model/sample.py:69-92. */
typedef struct seqdiff_config {
  int32_t hidden_size;         /* 768                                             */
  int32_t num_attention_heads; /* 12 (head_dim must be 64)                        */
  int32_t intermediate_size;   /* 1024                                            */
  int32_t num_hidden_layers;   /* 6                                               */
  int32_t max_position_embeddings; /* = max_seq_len; distance_embedding rows = 2P-1 */
  int32_t feature_size;        /* 20                                              */
  int32_t relative_key;        /* 1: position_embedding_type == "relative_key"    */
  float layer_norm_eps;        /* 1e-12                                           */
} seqdiff_config_t;

SEQDIFF_API int seqdiff_abi_version(void);
SEQDIFF_API const char* seqdiff_last_error(void);
/* number of kernels this library has launched in this process (bench.py's `gpu_launches`) */
SEQDIFF_API uint64_t seqdiff_launch_count(void);

/* built-in event profiler (bench.py roofline numbers): between begin and end every kernel this library
 * launches OUTSIDE graph capture is followed by a CUDA event on its stream; end() synchronises the device and
 * returns per-kernel-tag totals: tags[i*tag_stride..] (NUL-terminated), ms[i], counts[i]; result = #tags or <0. */
SEQDIFF_API int seqdiff_profile_begin(void* stream);
SEQDIFF_API int seqdiff_profile_end(char* tags, int tag_stride, float* ms, int* counts, int cap);
/* debug: device buffer of 4 x 1024 uint64 that CTA 0 of the pipelined attention kernel fills with its role timelines
 * (slot 0 of each role = event count, then (SM clock << 8 | event id)); NULL (default) switches tracing off. */
SEQDIFF_API int seqdiff_debug_attn_trace(void* device_buf);
/* debug build only (SEQDIFF_DEBUG_BOUNDS=1 python build.py -> libseqdiff_b200_dbg.so; the GPU pool does not allow compute-sanitizer):
 * every buffer carved out of a forward / sampling / training workspace is followed by a 256-byte guard band; this call waits for the
 * device and verifies all bands (error = some kernel wrote past the end of a buffer).  The product build has no bands: 0 / 0, OK. */
SEQDIFF_API int seqdiff_debug_check_guards(int* n_bands, int* n_broken, void* stream);

/* ---- model handle: replaces ConditionalBertForDiffusionBase.__init__ + load_state_dict ---------
 * sequence_model/model.py:156-181, sample.py:106.  Tensor names are the reference state_dict keys
 * (SURVEY.md Appendix B), e.g. "decoder.layer.0.attention.self.query.weight"; data is fp32. */
SEQDIFF_API int seqdiff_model_create(const seqdiff_config_t* cfg, int device, seqdiff_model_t** out);
SEQDIFF_API int seqdiff_model_destroy(seqdiff_model_t* m);
SEQDIFF_API int seqdiff_model_set_tensor(seqdiff_model_t* m, const char* name, const float* data, int64_t numel, void* stream);
/* packs fused QKV / cross-KV weights and the bf16 copies; must follow the last set_tensor */
SEQDIFF_API int seqdiff_model_finalize(seqdiff_model_t* m, void* stream);

/* ---- denoiser forward: replaces ConditionalBertForDiffusionBase.forward, model.py:200-237 --------
 * timestep [B] f32; noised_ligand_seq [B,L_lig,20]; ligand_angle [B,L_lig,8]; ligand_mask [B,L_lig]
 * ({0,1} floats); receptor_* likewise with L_rec; logits_out [B,L_lig,feature_size] f32. */
SEQDIFF_API int seqdiff_forward(seqdiff_model_t* m, int precision, int B, int L_lig, int L_rec, const float* timestep,
                    const float* noised_ligand_seq, const float* ligand_angle, const float* ligand_mask,
                    const float* receptor_seq, const float* receptor_angle, const float* receptor_mask,
                    float* logits_out, void* stream);

/* ---- reverse step: replaces sample_p_zs_given_zt_discrete (+ compute_batched_over0_posterior_
 * distribution), sequence_model/sample.py:120-179, for is_last_step == False.
 * q_tables [n_tab,3,20,20] f32 = (Qt, Qsb, Qtb) per graph (n_tab == B) or shared (n_tab == 1), built by
 * the host with the caller's noise_schedule/transition objects exactly as sample.py:156-160 does.
 * noise_E [B*L,20] = the Exp(1) race noise of torch.multinomial (parity mode) or NULL -> counter-based
 * Philox4x32-10 keyed by (seed, graph_id0 + b, residue, step).  diverse == 0 -> argmax.
 * x_s_out [B,L,20] one-hot f32 (may alias noised_data); idx_out [B*L] u8 or NULL. */
SEQDIFF_API int seqdiff_reverse_step(const float* q_tables, int n_tab, int B, int L, const float* noised_data,
                         const float* pred_logits, int diverse, const float* noise_E, uint64_t seed,
                         uint64_t graph_id0, uint32_t step, float* x_s_out, uint8_t* idx_out, void* stream);

/* ---- training q-sample: replaces PeptideDiff.apply_aa_noise, model.py:291-311 --------------------
 * qtb [B,20,20] f32 = get_Qt_bar(alpha_bar(t_int/T)); rows of x0 that are all-zero (padding) -> class 0. */
SEQDIFF_API int seqdiff_apply_aa_noise(const float* qtb, int B, int L, const float* x0, const float* noise_E, uint64_t seed,
                           uint64_t graph_id0, uint32_t step, float* x_t_out, uint8_t* idx_out, void* stream);

/* ---- batch collation: replaces LigandBindingSiteDataset.__getitem__, sequence_model/dataset.py:97-129 ----------
 * G complexes stored ragged: node_offsets [G+1] i32; ligand_mask, pocket_mask [total] u8; angle_features [total,8] f32;
 * amino_acid [total,20] f32 one-hot.  Pocket mask dilated by exactly +-pocket_ext with torch.roll wrap-around semantics
 * (quirk Q9), rows compacted in order, zero-padded to max_len; *_attn prefix-ones.  lengths [G,2] i32 = (n_lig, n_rec)
 * before clamping: a value > max_len is the reference's RuntimeError("Length exceed") (raised by the host wrapper). */
SEQDIFF_API int seqdiff_collate(int G, const int32_t* node_offsets, const uint8_t* ligand_mask, const uint8_t* pocket_mask,
                    const float* angle_features, const float* amino_acid, int pocket_ext, int max_len, float* ligand_angles,
                    float* ligand_seq, float* ligand_attn_mask, float* receptor_angles, float* receptor_seq,
                    float* receptor_attn_mask, int32_t* lengths, void* stream);

/* ---- whole reverse-diffusion loop: replaces the T-step loop of denoise(), sample.py:192-207 -------
 * q_tables_steps [T,3,20,20]: entry s holds (Qt,Qsb,Qtb) for the step s_int = s (t=(s+1)/T).
 * x_T [B,L_lig,20] one-hot start.  noise_E_steps [T,B*L_lig,20] (entry s used at step s; entry 0 unused)
 * or NULL -> Philox.  One step = forward + reverse step, replayed from a captured CUDA graph.
 * final_out [B,L_lig,20]: raw logits of the last step (quirk: sample.py:147-148). */
SEQDIFF_API int seqdiff_sample(seqdiff_model_t* m, int precision, int B, int L_lig, int L_rec, int T,
                   const float* q_tables_steps, const float* x_T, const float* ligand_angle,
                   const float* ligand_mask, const float* receptor_seq, const float* receptor_angle,
                   const float* receptor_mask, int diverse, const float* noise_E_steps, uint64_t seed,
                   uint64_t graph_id0, float* final_out, void* stream);

/* The same loop with options.  flags bit 0 (SEQDIFF_SAMPLE_PACKED): ragged packing -- only the valid prefix of every graph
 * (ligand_mask / receptor_mask must be prefixes of ones, as LigandBindingSiteDataset builds them, dataset.py:110-114) is carried
 * through the GEMMs / LayerNorms / attention: M = sum of lengths instead of B * L.  Results at valid positions are bit-identical
 * to the padded computation (a padded key's probability underflows to exactly 0, every other operator is row-local); the
 * reference also computes and samples the padded positions, which denoise() never reads (sample.py:211-224) -- here they
 * come back as 0 in final_out.  Non-prefix masks or fp32 mode silently take the padded path. */
#define SEQDIFF_SAMPLE_PACKED 1
SEQDIFF_API int seqdiff_sample_ex(seqdiff_model_t* m, int precision, int B, int L_lig, int L_rec, int T,
                      const float* q_tables_steps, const float* x_T, const float* ligand_angle,
                      const float* ligand_mask, const float* receptor_seq, const float* receptor_angle,
                      const float* receptor_mask, int diverse, const float* noise_E_steps, uint64_t seed,
                      uint64_t graph_id0, int flags, float* final_out, void* stream);

/* The same loop for P pockets x K samples per pocket (peptide design: many candidate sequences for one binding pocket).  Ligand-side
 * arrays hold B = P*K graphs, sample j of pocket p being graph p*K + j with global graph id graph_id0 + p*K + j in the Philox stream:
 * x_T / final_out [P*K,L_lig,20], ligand_angle [P*K,L_lig,8], ligand_mask [P*K,L_lig], noise_E_steps [T,P*K*L_lig,20] or NULL.
 * Receptor-side arrays hold the P pockets once: receptor_seq [P,L_rec,20], receptor_angle [P,L_rec,8], receptor_mask [P,L_rec].
 * The receptor rows of a step (angle embedding, ligand_feature_emb's adaLN + MLP, all decoder layers' cross K|V) depend on the
 * pocket and the step only, so they are computed once per pocket and the K samples' cross-attention reads them.  final_out equals,
 * bit for bit, what seqdiff_sample_ex returns for the batch whose receptor arrays are repeated K times per pocket (packed mode:
 * at the valid positions, padded ones 0).  K = 1 is seqdiff_sample_ex.  P < 1, K < 1 or P*K*max(L_lig, L_rec) > INT32_MAX:
 * SEQDIFF_ERR_INVALID. */
SEQDIFF_API int seqdiff_sample_multi(seqdiff_model_t* m, int precision, int P, int K, int L_lig, int L_rec, int T,
                         const float* q_tables_steps, const float* x_T, const float* ligand_angle,
                         const float* ligand_mask, const float* receptor_seq, const float* receptor_angle,
                         const float* receptor_mask, int diverse, const float* noise_E_steps, uint64_t seed,
                         uint64_t graph_id0, int flags, float* final_out, void* stream);

/* ---- output decode: replaces the per-graph loop of denoise(), sequence_model/sample.py:208-224 --------------------
 * final_seq [B,L,20] (the loop's result: raw logits of the last step), true_seq [B,L,20] one-hot, ligand_mask [B,L] {0,1}.
 * pred_idx / true_idx [B,L] u8 = argmax over classes (first maximum, like torch.argmax); counts [B,2] i32 =
 * (#masked positions where pred == true, #masked positions): recovery_rate = counts[b][0] / counts[b][1] (sample.py:214-216).
 * The host only joins AA_VOCAB letters over the masked prefix. */
SEQDIFF_API int seqdiff_decode(int B, int L, const float* final_seq, const float* true_seq, const float* ligand_mask, uint8_t* pred_idx,
                   uint8_t* true_idx, int32_t* counts, void* stream);

/* ---- loss terms (evaluation): replaces the reductions of PeptideDiff.get_loss, sequence_model/model.py:313-345, and
 * elbo_loss, sequence_model/utils.py:132-161, over N = B*L rows.  logits [N,20]; x0, x_t [N,20] one-hot; ligand_mask [N].
 * noised(n) = argmax(x_t[n]) != argmax(x0[n]); sel(n) = mask(n) && !noised(n).  terms [10] f64 (device):
 *   [0] #mask  [1] #noised  [2] #sel  [3] #(mask && argmax x_t == argmax x0)  [4] #(mask && argmax logits == argmax x0)
 *   [5] sum_{noised} CE(logits, x0)   [6] sum_{sel} CE(logits, x0)
 *   [7] sum_{noised} sum_c softmax(logits)_c * log_softmax(logits + 1e-6)_c          (nll = -[7] / [1])
 *   [8] sum_{noised} sum_c q_c * (log q_c - log_softmax(logits + 1e-6)_c), q = softmax(x0)   (kl_div batchmean = [8] / [1])
 *   [9] reserved (0).
 * total_loss = [5]/[1] + (-[7]/[1] + [8]/[1]).  Backward is not part of this library. */
SEQDIFF_API int seqdiff_loss_terms(int N, const float* logits, const float* x0, const float* x_t, const float* ligand_mask, double* terms,
                       void* stream);

/* ==== training step: BASELINE configs[3] ("sequence_model training step batch 128 graphs with NCCL gradient allreduce") ==========
 * Replaces, for one optimizer step, autograd over PeptideDiff.training_step / get_loss (sequence_model/model.py:313-367),
 * torch.optim.AdamW (model.py:420-422; lr 5e-5, weight_decay 0.1: train_model.py:30-31) and Lightning's gradient_clip_val = 1.0
 * (train_model.py:33,95).  The library never communicates: a data-parallel caller all-reduces the flat gradient buffer between
 * seqdiff_train_step and seqdiff_adamw_step (train.py does that with torch.distributed / NCCL).
 *
 * Trainable tensors = the state_dict of ConditionalBertForDiffusionBase minus the `timestep_projector.W` buffer and minus
 * `receptor_feature_emb.*`, which the reference never uses (model.py:221) and whose .grad therefore stays None.  They are laid out
 * in ONE flat fp32 index space (gradients, AdamW moments); seqdiff_train_param_table returns the (name, offset, numel) triples. */
SEQDIFF_API int64_t seqdiff_train_param_count(seqdiff_model_t* m);   /* elements of the flat buffers, or -1 */
/* names[i*name_stride..] (NUL-terminated), offsets[i], numels[i]; returns the number of tensors (call with cap = 0 to query it) */
SEQDIFF_API int seqdiff_train_param_table(seqdiff_model_t* m, char* names, int name_stride, int64_t* offsets, int64_t* numels, int cap);
/* Overlap of the data-parallel all-reduce with the backward pass.  The flat index space follows the forward order of the network, so
 * the backward pass finishes it from the end: seqdiff_train_grad_buckets returns n and bounds[0..n] (ascending offsets, bucket k =
 * [bounds[k], bounds[k+1])); bucket n-1 (decoder_normalize + head) is final first, bucket 0 (embeddings + ligand_feature_emb) last.
 * seqdiff_train_set_bucket_events registers n caller-owned cudaEvent_t (NULL entries allowed; n = 0 clears): every following
 * seqdiff_train_step records event k on its stream as soon as bucket k holds its final gradients, so a communication stream can
 * wait on it and reduce that range while the rest of the backward pass runs (train.py: FlatAdamW).  Replaces what DDP's gradient
 * hooks + bucketing do under Lightning for the reference (train_model.py:92-110). */
SEQDIFF_API int seqdiff_train_grad_buckets(seqdiff_model_t* m, int64_t* bounds, int cap);  /* returns n (cap = 0: query), -1 on error */
SEQDIFF_API int seqdiff_train_set_bucket_events(seqdiff_model_t* m, void** events, int n);
/* forward (training mode) + loss + backward.  t_norm [B] = t_int / T as the reference passes it when training (quirk Q3);
 * noised_ligand_seq = apply_aa_noise(ligand_seq, t_int) (seqdiff_apply_aa_noise); ligand_seq [B,L_lig,20] one-hot targets.
 * p_hidden / p_attn = hidden_dropout_prob / attention_probs_dropout_prob (0 for parity runs); masks come from Philox keyed by
 * (seed, dropout site, element, step).  grads_out: flat fp32 [param_count], overwritten with d(total_loss)/d(theta) for
 * total_loss = CrossEntropy(noised rows) + elbo_loss(noised rows) (model.py:330-344).  loss_terms_out: double[10] on the device,
 * layout of seqdiff_loss_terms.  logits_out (optional) [B,L_lig,20].  L_lig, L_rec <= 128 and B*L % 8 == 0. */
SEQDIFF_API int seqdiff_train_step(seqdiff_model_t* m, int precision, int B, int L_lig, int L_rec, const float* t_norm,
                       const float* noised_ligand_seq, const float* ligand_seq, const float* ligand_angle, const float* ligand_mask,
                       const float* receptor_seq, const float* receptor_angle, const float* receptor_mask, float p_hidden, float p_attn,
                       uint64_t seed, uint32_t step, float* grads_out, double* loss_terms_out, float* logits_out, void* stream);
/* g <- grad_scale * grads (grad_scale = 1 / world after a summing all-reduce); clip_grad_norm_(max_grad_norm) (<= 0: off);
 * AdamW step `step` (1-based) on the handle's fp32 master weights with moments exp_avg / exp_avg_sq (flat fp32, zero-initialised
 * by the caller); then the packed operand copies are refreshed in place.  grad_norm_out (optional, device): pre-clip global norm. */
SEQDIFF_API int seqdiff_adamw_step(seqdiff_model_t* m, const float* grads, float* exp_avg, float* exp_avg_sq, float grad_scale,
                       float max_grad_norm, float lr, float beta1, float beta2, float eps, float weight_decay, int step,
                       float* grad_norm_out, void* stream);
/* copies a master tensor out of the handle (checkpointing / tests): state_dict name -> fp32 [numel] */
SEQDIFF_API int seqdiff_model_get_tensor(seqdiff_model_t* m, const char* name, float* out, int64_t numel, void* stream);

/* ==== structure (angle) model: SURVEY.md section 8(f) row 3 ===========================================================
 * Same handle type and the same set_tensor / finalize / destroy calls; tensor names are the state_dict keys of
 * structure_model/model.py:163-178 ("receptor_seq_emb.linear.weight", "encoder.layer.0.attention.self.query.weight",
 * "timestep_emb.adaLN_modulation.2.weight", "angles_predictor.dense2.bias", ...).  cfg.feature_size = number of angle
 * features (8); encoder and decoder share every other BertConfig field (structure_model/sample.py:151-173). */
SEQDIFF_API int seqdiff_struct_model_create(const seqdiff_config_t* cfg, int device, seqdiff_model_t** out);

/* replaces ConditionalBertForDiffusionBase.forward, structure_model/model.py:180-215.
 * timestep [B] f32 (the reference passes int64 step indices; the product t * W is formed in fp32 either way);
 * noised_ligand_angles [B,L_lig,F]; ligand_mask [B,L_lig]; receptor_seq [B,L_rec,20]; receptor_angles [B,L_rec,F];
 * receptor_mask [B,L_rec]; out [B,L_lig,F] f32 (predicted noise). */
SEQDIFF_API int seqdiff_struct_forward(seqdiff_model_t* m, int precision, int B, int L_lig, int L_rec, const float* timestep,
                           const float* noised_ligand_angles, const float* ligand_mask, const float* receptor_seq,
                           const float* receptor_angles, const float* receptor_mask, float* out, void* stream);

/* replaces the arithmetic of p_sample after the model call (structure_model/sample.py:92-101) plus, when wrap != 0, the angle
 * wrap of p_sample_loop (sample.py:139-141; utils.py:20-40).  coef_steps [T,4] f32 = per step index
 * (1/sqrt(alpha_t), beta_t, sqrt(1 - alphabar_t), sqrt(posterior_variance_t)), built by the host from compute_alphas(betas).
 * noise [B*L*F] N(0,1) (what torch.randn_like drew) or NULL -> Philox4x32-10 + Box-Muller keyed by
 * (seed, graph_id0 + b, element group, step); ignored at step 0.  x_out may alias x_t. */
SEQDIFF_API int seqdiff_struct_p_sample(const float* coef_steps, int T, int step, int B, int L, int F, const float* x_t,
                            const float* model_output, const float* noise, uint64_t seed, uint64_t graph_id0, int wrap,
                            float* x_out, void* stream);

/* replaces p_sample_loop, structure_model/sample.py:104-144 (STEP = 1): steps T-1 .. 0, each = forward + p_sample + wrap.
 * The receptor branch does not depend on the step and is evaluated once.  noise_steps [T, B*L_lig*F] (entry i used at step
 * index i; entry 0 unused) or NULL -> Philox.  steps_out [T, B*L_lig*F] or NULL: entry k = angles after the k-th reverse step
 * (the tensor the reference returns); final_out [B,L_lig,F] = its last entry. */
SEQDIFF_API int seqdiff_struct_sample(seqdiff_model_t* m, int precision, int B, int L_lig, int L_rec, int T, const float* coef_steps,
                          const float* x_T, const float* ligand_mask, const float* receptor_seq, const float* receptor_angles,
                          const float* receptor_mask, const float* noise_steps, uint64_t seed, uint64_t graph_id0,
                          float* steps_out, float* final_out, void* stream);

/* ---- operator-level entry points (used by the parity tests and the micro benchmarks) --------------
 * C[M,N] = epilogue(A[M,K] * W[N,K]^T + bias[N] (+ resid[M,N])); epilogue: 0 none, 1 erf-GELU, 2 SiLU.
 * precision FP32: all f32 (SIMT kernel).  BF16 / FP16: A and W are 16-bit in the mode's formats
 * (tcgen05 + TMA kernel); resid (optional) is f32 and makes C f32, otherwise C has A's 16-bit type. */
SEQDIFF_API int seqdiff_op_gemm(int precision, int M, int N, int K, const void* A, const void* W, const float* bias,
                    const void* resid, int epilogue, void* C, void* stream);
/* Linear + residual + the LayerNorm that follows it (HF BertSelfOutput / BertOutput, modeling_bert: dense -> dropout ->
 * LayerNorm(hidden + input)) in one launch, 16-bit modes only, N in {512, 768, 1024}:
 *   C[M,N] (f32) = A * W^T + bias + resid ;  h[M,N] (16-bit) = LayerNorm(C) * ln_w + ln_b ;  stats[M] = (mean, rstd) as float2 */
SEQDIFF_API int seqdiff_op_gemm_ln(int precision, int M, int N, int K, const void* A, const void* W, const float* bias,
                       const float* resid, const float* ln_w, const float* ln_b, float eps, float* C, void* h, float* stats,
                       void* stream);
/* multi-head attention core of HF BertSelfAttention (4.38.2 relative_key semantics, SURVEY.md App. A):
 * q [B,Lq,*] k,v [B,Lk,*] with row strides (elements) ldq/ldk/ldv, heads x 64; dist_emb [2P-1,64] or NULL;
 * key_mask [B,Lk] {0,1} -> additive (1-m)*-10000; out [B,Lq,heads*64].  Element type by precision. */
SEQDIFF_API int seqdiff_op_attention(int precision, int B, int heads, int Lq, int Lk, const void* q, int ldq, const void* k,
                         int ldk, const void* v, int ldv, const void* dist_emb, int P, const float* key_mask,
                         void* out, void* stream);
/* training attention (csrc/attention_train*.cu): the attention core above with dropout on the probabilities (mask from Philox keyed by
 * (seed, site, element, step); p_drop = 0: none), and its backward.  impl 0: warp-level tensor-core kernels (16-bit modes only),
 * 1: fp32 SIMT kernels (all modes; the fp32 parity path).  L <= 128.  out / dout / dq / dk / dv: [B, L, heads*64] dense;
 * dE [2P-1, 64] f32 is ACCUMULATED into (zero it first); NULL when dist_emb is NULL. */
/* C[M,N] (+)= At^T Bt: At [K,M], Bt [K,N] row-major 16-bit, C fp32 (pre-zeroed when split_k != 1; split_k = -1: auto).  The weight-gradient
 * product of the training step with both operands MN-major for tcgen05 (no transposed copies).  Operator-level entry for tests. */
SEQDIFF_API int seqdiff_op_gemm_tn(int precision, int M, int N, int K, const void* At, const void* Bt, float* C, int split_k, void* stream);
SEQDIFF_API int seqdiff_op_attention_train_fwd(int precision, int impl, int B, int heads, int Lq, int Lk, const void* q, int ldq, const void* k,
                                   int ldk, const void* v, int ldv, const void* dist_emb, int P, const float* key_mask, float p_drop,
                                   uint64_t seed, uint32_t site, uint32_t step, void* out, void* stream);
SEQDIFF_API int seqdiff_op_attention_train_bwd(int precision, int impl, int B, int heads, int Lq, int Lk, const void* q, int ldq, const void* k,
                                   int ldk, const void* v, int ldv, const void* dist_emb, int P, const float* key_mask, float p_drop,
                                   uint64_t seed, uint32_t site, uint32_t step, const void* dout, void* dq, void* dk, void* dv, float* dE,
                                   void* stream);
/* post-LN of HF BertSelfOutput / BertOutput: y = LayerNorm(in) * ln_w + ln_b over rows of H (256/512/768/1024) fp32 values.
 * out32 [M,H] f32 and/or out16 [M,H] in the mode's 16-bit format (either may be NULL); stats [M] (mean, rstd) float2 or NULL. */
SEQDIFF_API int seqdiff_op_layernorm(int precision, int M, int H, const float* in, const float* ln_w, const float* ln_b, float eps,
                         float* out32, void* out16, float* stats, void* stream);
/* Philox4x32-10 stream the sampler uses: out[n*20+j] = raw u32 for (seed, graph, residue, step, class) */
SEQDIFF_API int seqdiff_op_philox_u32(uint64_t seed, uint64_t graph_id0, uint32_t step, int B, int L, uint32_t* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SEQDIFF_B200_H_ */
