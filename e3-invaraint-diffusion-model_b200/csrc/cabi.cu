// cabi.cu -- the extern "C" surface declared in include/seqdiff_b200.h.  Thin: argument checks, handle
// casts, exception firewall.  No torch types, no allocation on behalf of the caller.
#include <cstdio>
#include <new>

#include "model.cuh"

namespace seqdiff {
const char* last_error();
}
using namespace seqdiff;

#define SD_GUARD_BEGIN try {
#define SD_GUARD_END                                         \
  }                                                          \
  catch (const std::exception& e) {                          \
    set_error(std::string("exception: ") + e.what());        \
    return SEQDIFF_ERR_STATE;                                \
  }                                                          \
  catch (...) {                                              \
    set_error("unknown exception");                          \
    return SEQDIFF_ERR_STATE;                                \
  }

struct seqdiff_model {
  Model impl;
};

extern "C" {

int seqdiff_abi_version(void) { return SEQDIFF_ABI_VERSION; }
const char* seqdiff_last_error(void) { return last_error(); }
uint64_t seqdiff_launch_count(void) { return g_launches.load(); }

int seqdiff_profile_begin(void* stream) {
  SD_GUARD_BEGIN
  return profile_begin(static_cast<cudaStream_t>(stream));
  SD_GUARD_END
}
int seqdiff_profile_end(char* tags, int tag_stride, float* ms, int* counts, int cap) {
  if (!tags || !ms || !counts || tag_stride < 8 || cap < 1) return -1;
  return profile_end(tags, tag_stride, ms, counts, cap);
}

int seqdiff_debug_attn_trace(void* device_buf) {
  g_attn_trace = static_cast<unsigned long long*>(device_buf);
  return SEQDIFF_OK;
}

int seqdiff_debug_check_guards(int* n_bands, int* n_broken, void* stream) {
  SD_GUARD_BEGIN
  int nb = 0, nk = 0;
  SD_TRY(debug_guard_check(static_cast<cudaStream_t>(stream), &nb, &nk));
  if (n_bands) *n_bands = nb;
  if (n_broken) *n_broken = nk;
  if (nk) {
    set_error(std::to_string(nk) + " of " + std::to_string(nb) + " workspace guard bands were overwritten (out-of-bounds write past a carved buffer)");
    return SEQDIFF_ERR_STATE;
  }
  return SEQDIFF_OK;
  SD_GUARD_END
}

int seqdiff_model_create(const seqdiff_config_t* cfg, int device, seqdiff_model_t** out) {
  SD_GUARD_BEGIN
  SD_CHECK(cfg != nullptr && out != nullptr, "null argument");
  int ndev = 0;
  SD_CUDA(cudaGetDeviceCount(&ndev));
  SD_CHECK(device >= 0 && device < ndev, "no such CUDA device");
  seqdiff_model* m = new (std::nothrow) seqdiff_model();
  SD_CHECK(m != nullptr, "out of host memory");
  const int rc = m->impl.init(*cfg, device);
  if (rc != SEQDIFF_OK) {
    delete m;
    return rc;
  }
  *out = m;
  return SEQDIFF_OK;
  SD_GUARD_END
}

int seqdiff_model_destroy(seqdiff_model_t* m) {
  SD_GUARD_BEGIN
  if (m) {
    cudaSetDevice(m->impl.device);
    cudaDeviceSynchronize();
    delete m;
  }
  return SEQDIFF_OK;
  SD_GUARD_END
}

int seqdiff_model_set_tensor(seqdiff_model_t* m, const char* name, const float* data, int64_t numel, void* stream) {
  SD_GUARD_BEGIN
  SD_CHECK(m && name && data, "null argument");
  return m->impl.set_tensor(name, data, numel, static_cast<cudaStream_t>(stream));
  SD_GUARD_END
}

int seqdiff_model_finalize(seqdiff_model_t* m, void* stream) {
  SD_GUARD_BEGIN
  SD_CHECK(m, "null argument");
  return m->impl.finalize(static_cast<cudaStream_t>(stream));
  SD_GUARD_END
}

int seqdiff_forward(seqdiff_model_t* m, int precision, int B, int L_lig, int L_rec, const float* timestep,
                    const float* noised_ligand_seq, const float* ligand_angle, const float* ligand_mask,
                    const float* receptor_seq, const float* receptor_angle, const float* receptor_mask, float* logits_out,
                    void* stream) {
  SD_GUARD_BEGIN
  SD_CHECK(m && timestep && noised_ligand_seq && ligand_angle && ligand_mask && receptor_seq && receptor_angle && receptor_mask &&
               logits_out,
           "null argument");
  return m->impl.forward(precision, B, L_lig, L_rec, timestep, nullptr, noised_ligand_seq, ligand_angle, ligand_mask, receptor_seq,
                         receptor_angle, receptor_mask, logits_out, static_cast<cudaStream_t>(stream));
  SD_GUARD_END
}

int seqdiff_reverse_step(const float* q_tables, int n_tab, int B, int L, const float* noised_data, const float* pred_logits,
                         int diverse, const float* noise_E, uint64_t seed, uint64_t graph_id0, uint32_t step, float* x_s_out,
                         uint8_t* idx_out, void* stream) {
  SD_GUARD_BEGIN
  SD_CHECK(q_tables && noised_data && pred_logits && x_s_out, "null argument");
  return reverse_step(q_tables, n_tab, B, L, noised_data, pred_logits, diverse, noise_E, seed, graph_id0, step, nullptr, x_s_out,
                      idx_out, static_cast<cudaStream_t>(stream));
  SD_GUARD_END
}

int seqdiff_apply_aa_noise(const float* qtb, int B, int L, const float* x0, const float* noise_E, uint64_t seed,
                           uint64_t graph_id0, uint32_t step, float* x_t_out, uint8_t* idx_out, void* stream) {
  SD_GUARD_BEGIN
  SD_CHECK(qtb && x0 && x_t_out, "null argument");
  return apply_aa_noise(qtb, B, L, x0, noise_E, seed, graph_id0, step, x_t_out, idx_out, static_cast<cudaStream_t>(stream));
  SD_GUARD_END
}

int seqdiff_collate(int G, const int32_t* node_offsets, const uint8_t* ligand_mask, const uint8_t* pocket_mask,
                    const float* angle_features, const float* amino_acid, int pocket_ext, int max_len, float* ligand_angles,
                    float* ligand_seq, float* ligand_attn_mask, float* receptor_angles, float* receptor_seq, float* receptor_attn_mask,
                    int32_t* lengths, void* stream) {
  SD_GUARD_BEGIN
  SD_CHECK(node_offsets && ligand_mask && pocket_mask && angle_features && amino_acid && ligand_angles && ligand_seq && ligand_attn_mask &&
               receptor_angles && receptor_seq && receptor_attn_mask && lengths,
           "null argument");
  SD_CHECK(pocket_ext >= 0, "pocket_ext must be >= 0");
  return collate(G, node_offsets, ligand_mask, pocket_mask, angle_features, amino_acid, pocket_ext, max_len, ligand_angles, ligand_seq,
                 ligand_attn_mask, receptor_angles, receptor_seq, receptor_attn_mask, lengths, static_cast<cudaStream_t>(stream));
  SD_GUARD_END
}

int seqdiff_sample(seqdiff_model_t* m, int precision, int B, int L_lig, int L_rec, int T, const float* q_tables_steps,
                   const float* x_T, const float* ligand_angle, const float* ligand_mask, const float* receptor_seq,
                   const float* receptor_angle, const float* receptor_mask, int diverse, const float* noise_E_steps,
                   uint64_t seed, uint64_t graph_id0, float* final_out, void* stream) {
  SD_GUARD_BEGIN
  SD_CHECK(m && q_tables_steps && x_T && ligand_angle && ligand_mask && receptor_seq && receptor_angle && receptor_mask && final_out,
           "null argument");
  return m->impl.sample(precision, B, 1, L_lig, L_rec, T, q_tables_steps, x_T, ligand_angle, ligand_mask, receptor_seq, receptor_angle,
                        receptor_mask, diverse, noise_E_steps, seed, graph_id0, final_out, static_cast<cudaStream_t>(stream));
  SD_GUARD_END
}

int64_t seqdiff_train_param_count(seqdiff_model_t* m) {
  try {
    if (!m) return -1;
    return m->impl.train_param_count();
  } catch (...) {
    return -1;
  }
}

int seqdiff_train_param_table(seqdiff_model_t* m, char* names, int name_stride, int64_t* offsets, int64_t* numels, int cap) {
  try {
    if (!m || m->impl.build_slots() != SEQDIFF_OK) return -1;
    const int n = static_cast<int>(m->impl.slots.size());
    if (cap <= 0) return n;
    if (!names || !offsets || !numels || name_stride < 16) return -1;
    for (int i = 0; i < n && i < cap; ++i) {
      std::snprintf(names + static_cast<size_t>(i) * name_stride, name_stride, "%s", m->impl.slots[i].name.c_str());
      offsets[i] = m->impl.slots[i].off;
      numels[i] = m->impl.slots[i].numel;
    }
    return n;
  } catch (...) {
    return -1;
  }
}

int seqdiff_train_grad_buckets(seqdiff_model_t* m, int64_t* bounds, int cap) {
  try {
    if (!m || m->impl.build_slots() != SEQDIFF_OK) return -1;
    const int n = static_cast<int>(m->impl.grad_bucket_bounds.size()) - 1;
    if (cap <= 0) return n;
    if (!bounds || cap < n + 1) return -1;
    for (int i = 0; i <= n; ++i) bounds[i] = m->impl.grad_bucket_bounds[i];
    return n;
  } catch (...) {
    return -1;
  }
}

int seqdiff_train_set_bucket_events(seqdiff_model_t* m, void** events, int n) {
  SD_GUARD_BEGIN
  SD_CHECK(m && n >= 0 && (n == 0 || events), "null argument");
  SD_TRY(m->impl.build_slots());
  SD_CHECK(n == 0 || n == static_cast<int>(m->impl.grad_bucket_bounds.size()) - 1, "one event slot per gradient bucket (seqdiff_train_grad_buckets)");
  m->impl.bucket_events.assign(static_cast<size_t>(n), nullptr);
  for (int i = 0; i < n; ++i) m->impl.bucket_events[i] = static_cast<cudaEvent_t>(events[i]);
  return SEQDIFF_OK;
  SD_GUARD_END
}

int seqdiff_train_step(seqdiff_model_t* m, int precision, int B, int L_lig, int L_rec, const float* t_norm, const float* noised_ligand_seq,
                       const float* ligand_seq, const float* ligand_angle, const float* ligand_mask, const float* receptor_seq,
                       const float* receptor_angle, const float* receptor_mask, float p_hidden, float p_attn, uint64_t seed, uint32_t step,
                       float* grads_out, double* loss_terms_out, float* logits_out, void* stream) {
  SD_GUARD_BEGIN
  SD_CHECK(m && t_norm && noised_ligand_seq && ligand_seq && ligand_angle && ligand_mask && receptor_seq && receptor_angle && receptor_mask &&
               grads_out && loss_terms_out,
           "null argument");
  TrainArgs a{};
  a.precision = precision; a.B = B; a.Ll = L_lig; a.Lr = L_rec;
  a.t_norm = t_norm; a.x_t = noised_ligand_seq; a.x0 = ligand_seq; a.lig_angle = ligand_angle; a.lig_mask = ligand_mask;
  a.rec_seq = receptor_seq; a.rec_angle = receptor_angle; a.rec_mask = receptor_mask;
  a.p_hidden = p_hidden; a.p_attn = p_attn; a.seed = seed; a.step = step;
  a.grads = grads_out; a.terms = loss_terms_out; a.logits_out = logits_out;
  return m->impl.train_step(a, static_cast<cudaStream_t>(stream));
  SD_GUARD_END
}

int seqdiff_adamw_step(seqdiff_model_t* m, const float* grads, float* exp_avg, float* exp_avg_sq, float grad_scale, float max_grad_norm, float lr,
                       float beta1, float beta2, float eps, float weight_decay, int step, float* grad_norm_out, void* stream) {
  SD_GUARD_BEGIN
  SD_CHECK(m && grads && exp_avg && exp_avg_sq, "null argument");
  return m->impl.adamw(grads, exp_avg, exp_avg_sq, grad_scale, max_grad_norm, lr, beta1, beta2, eps, weight_decay, step, grad_norm_out,
                       static_cast<cudaStream_t>(stream));
  SD_GUARD_END
}

int seqdiff_model_get_tensor(seqdiff_model_t* m, const char* name, float* out, int64_t numel, void* stream) {
  SD_GUARD_BEGIN
  SD_CHECK(m && name && out, "null argument");
  return m->impl.get_tensor(name, out, numel, static_cast<cudaStream_t>(stream));
  SD_GUARD_END
}

int seqdiff_sample_ex(seqdiff_model_t* m, int precision, int B, int L_lig, int L_rec, int T, const float* q_tables_steps, const float* x_T,
                      const float* ligand_angle, const float* ligand_mask, const float* receptor_seq, const float* receptor_angle,
                      const float* receptor_mask, int diverse, const float* noise_E_steps, uint64_t seed, uint64_t graph_id0, int flags,
                      float* final_out, void* stream) {
  SD_GUARD_BEGIN
  SD_CHECK(m && q_tables_steps && x_T && ligand_angle && ligand_mask && receptor_seq && receptor_angle && receptor_mask && final_out,
           "null argument");
  SD_CHECK((flags & ~1) == 0, "unknown sampling flag");
  return m->impl.sample(precision, B, 1, L_lig, L_rec, T, q_tables_steps, x_T, ligand_angle, ligand_mask, receptor_seq, receptor_angle,
                        receptor_mask, diverse, noise_E_steps, seed, graph_id0, final_out, static_cast<cudaStream_t>(stream), flags);
  SD_GUARD_END
}

int seqdiff_sample_multi(seqdiff_model_t* m, int precision, int P, int K, int L_lig, int L_rec, int T, const float* q_tables_steps,
                         const float* x_T, const float* ligand_angle, const float* ligand_mask, const float* receptor_seq,
                         const float* receptor_angle, const float* receptor_mask, int diverse, const float* noise_E_steps, uint64_t seed,
                         uint64_t graph_id0, int flags, float* final_out, void* stream) {
  SD_GUARD_BEGIN
  SD_CHECK(m && q_tables_steps && x_T && ligand_angle && ligand_mask && receptor_seq && receptor_angle && receptor_mask && final_out,
           "null argument");
  SD_CHECK(P >= 1 && K >= 1, "need at least one pocket and one sample per pocket");
  SD_CHECK(L_lig > 0 && L_rec > 0 && static_cast<int64_t>(P) * K * (L_lig > L_rec ? L_lig : L_rec) <= INT32_MAX,
           "pockets x samples x length overflows the row counts");
  SD_CHECK((flags & ~1) == 0, "unknown sampling flag");
  return m->impl.sample(precision, P, K, L_lig, L_rec, T, q_tables_steps, x_T, ligand_angle, ligand_mask, receptor_seq, receptor_angle,
                        receptor_mask, diverse, noise_E_steps, seed, graph_id0, final_out, static_cast<cudaStream_t>(stream), flags);
  SD_GUARD_END
}

int seqdiff_struct_model_create(const seqdiff_config_t* cfg, int device, seqdiff_model_t** out) {
  SD_GUARD_BEGIN
  SD_CHECK(cfg != nullptr && out != nullptr, "null argument");
  int ndev = 0;
  SD_CUDA(cudaGetDeviceCount(&ndev));
  SD_CHECK(device >= 0 && device < ndev, "no such CUDA device");
  seqdiff_model* m = new (std::nothrow) seqdiff_model();
  SD_CHECK(m != nullptr, "out of host memory");
  const int rc = m->impl.init(*cfg, device, kArchStructure);
  if (rc != SEQDIFF_OK) {
    delete m;
    return rc;
  }
  *out = m;
  return SEQDIFF_OK;
  SD_GUARD_END
}

int seqdiff_struct_forward(seqdiff_model_t* m, int precision, int B, int L_lig, int L_rec, const float* timestep,
                           const float* noised_ligand_angles, const float* ligand_mask, const float* receptor_seq,
                           const float* receptor_angles, const float* receptor_mask, float* out, void* stream) {
  SD_GUARD_BEGIN
  SD_CHECK(m && timestep && noised_ligand_angles && ligand_mask && receptor_seq && receptor_angles && receptor_mask && out, "null argument");
  return m->impl.struct_forward(precision, B, L_lig, L_rec, timestep, nullptr, noised_ligand_angles, ligand_mask, receptor_seq, receptor_angles,
                                receptor_mask, out, 3, static_cast<cudaStream_t>(stream));
  SD_GUARD_END
}

int seqdiff_struct_p_sample(const float* coef_steps, int T, int step, int B, int L, int F, const float* x_t, const float* model_output,
                            const float* noise, uint64_t seed, uint64_t graph_id0, int wrap, float* x_out, void* stream) {
  SD_GUARD_BEGIN
  SD_CHECK(coef_steps && x_t && model_output && x_out, "null argument");
  SD_CHECK(B > 0 && L > 0 && F > 0, "empty batch");
  return gauss_step(coef_steps, T, B, L * F, x_t, model_output, noise, seed, graph_id0, step, nullptr, x_out, nullptr,
                    static_cast<cudaStream_t>(stream), nullptr, wrap != 0);
  SD_GUARD_END
}

int seqdiff_struct_sample(seqdiff_model_t* m, int precision, int B, int L_lig, int L_rec, int T, const float* coef_steps, const float* x_T,
                          const float* ligand_mask, const float* receptor_seq, const float* receptor_angles, const float* receptor_mask,
                          const float* noise_steps, uint64_t seed, uint64_t graph_id0, float* steps_out, float* final_out, void* stream) {
  SD_GUARD_BEGIN
  SD_CHECK(m && coef_steps && x_T && ligand_mask && receptor_seq && receptor_angles && receptor_mask && final_out, "null argument");
  return m->impl.struct_sample(precision, B, L_lig, L_rec, T, coef_steps, x_T, ligand_mask, receptor_seq, receptor_angles, receptor_mask,
                               noise_steps, seed, graph_id0, steps_out, final_out, static_cast<cudaStream_t>(stream));
  SD_GUARD_END
}

int seqdiff_decode(int B, int L, const float* final_seq, const float* true_seq, const float* ligand_mask, uint8_t* pred_idx,
                   uint8_t* true_idx, int32_t* counts, void* stream) {
  SD_GUARD_BEGIN
  SD_CHECK(final_seq && true_seq && ligand_mask && pred_idx && true_idx && counts, "null argument");
  return decode_sequences(B, L, final_seq, true_seq, ligand_mask, pred_idx, true_idx, counts, static_cast<cudaStream_t>(stream));
  SD_GUARD_END
}

int seqdiff_loss_terms(int N, const float* logits, const float* x0, const float* x_t, const float* ligand_mask, double* terms, void* stream) {
  SD_GUARD_BEGIN
  SD_CHECK(logits && x0 && x_t && ligand_mask && terms, "null argument");
  return loss_terms(N, logits, x0, x_t, ligand_mask, terms, static_cast<cudaStream_t>(stream));
  SD_GUARD_END
}

int seqdiff_op_gemm(int precision, int M, int N, int K, const void* A, const void* W, const float* bias, const void* resid,
                    int epilogue, void* C, void* stream) {
  SD_GUARD_BEGIN
  SD_CHECK(A && W && bias && C, "null argument");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  // upper bits of `precision` may force the tile configuration (tests / sweeps): mode | (bn << 8) | (cta_pair << 20)
  const int force_bn = ((precision >> 8) & 0xfff) | (((precision >> 20) & 1) << 16);
  const int mode = precision & 0xff;
  if (mode == SEQDIFF_FP32)
    return gemm_f32(M, N, K, static_cast<const float*>(A), static_cast<const float*>(W), bias, static_cast<const float*>(resid),
                    epilogue, static_cast<float*>(C), s);
  SD_CHECK(mode == SEQDIFF_BF16 || mode == SEQDIFF_FP16, "bad precision");
  const int a_fmt = mode == SEQDIFF_FP16 ? 0 : 1;
  const int w_fmt = a_fmt;
  return gemm_16(M, N, K, A, a_fmt, W, w_fmt, bias, static_cast<const float*>(resid), epilogue, C, resid ? 2 : a_fmt, s, force_bn);
  SD_GUARD_END
}

int seqdiff_op_gemm_ln(int precision, int M, int N, int K, const void* A, const void* W, const float* bias, const float* resid,
                       const float* ln_w, const float* ln_b, float eps, float* C, void* h, float* stats, void* stream) {
  SD_GUARD_BEGIN
  SD_CHECK(A && W && bias && resid && ln_w && ln_b && C && h && stats, "null argument");
  SD_CHECK(precision == SEQDIFF_BF16 || precision == SEQDIFF_FP16, "fused GEMM + LayerNorm exists in the 16-bit modes only");
  const int fmt = precision == SEQDIFF_FP16 ? 0 : 1;
  const LnOut lo{ln_w, ln_b, eps, h, reinterpret_cast<float2*>(stats)};
  return gemm_16(M, N, K, A, fmt, W, fmt, bias, resid, 0, C, 2, static_cast<cudaStream_t>(stream), 0, nullptr, &lo);
  SD_GUARD_END
}

int seqdiff_op_attention(int precision, int B, int heads, int Lq, int Lk, const void* q, int ldq, const void* k, int ldk,
                         const void* v, int ldv, const void* dist_emb, int P, const float* key_mask, void* out, void* stream) {
  SD_GUARD_BEGIN
  SD_CHECK(q && k && v && key_mask && out, "null argument");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (precision == SEQDIFF_FP32)
    return attention<float>(B, heads, Lq, Lk, static_cast<const float*>(q), ldq, static_cast<const float*>(k), ldk,
                            static_cast<const float*>(v), ldv, static_cast<const float*>(dist_emb), P, key_mask,
                            static_cast<float*>(out), s);
  if (precision == SEQDIFF_FP16)
    return attention<f16>(B, heads, Lq, Lk, static_cast<const f16*>(q), ldq, static_cast<const f16*>(k), ldk,
                          static_cast<const f16*>(v), ldv, static_cast<const f16*>(dist_emb), P, key_mask, static_cast<f16*>(out), s);
  SD_CHECK(precision == SEQDIFF_BF16, "bad precision");
  return attention<bf16>(B, heads, Lq, Lk, static_cast<const bf16*>(q), ldq, static_cast<const bf16*>(k), ldk,
                         static_cast<const bf16*>(v), ldv, static_cast<const bf16*>(dist_emb), P, key_mask, static_cast<bf16*>(out), s);
  SD_GUARD_END
}

// training attention, operator level: impl 0 = wmma tensor-core kernels (16-bit modes), 1 = fp32 SIMT kernels (every mode),
// 2 (forward only) = the pipelined tcgen05 kernel with in-kernel dropout
int seqdiff_op_attention_train_fwd(int precision, int impl, int B, int heads, int Lq, int Lk, const void* q, int ldq, const void* k, int ldk,
                                   const void* v, int ldv, const void* dist_emb, int P, const float* key_mask, float p_drop, uint64_t seed,
                                   uint32_t site, uint32_t step, void* out, void* stream) {
  SD_GUARD_BEGIN
  SD_CHECK(q && k && v && key_mask && out, "null argument");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const DropSpec dr{p_drop, site, step, seed};
#define SD_ATF(T, FN) FN<T>(B, heads, Lq, Lk, static_cast<const T*>(q), ldq, static_cast<const T*>(k), ldk, static_cast<const T*>(v), ldv, \
                           static_cast<const T*>(dist_emb), P, key_mask, dr, static_cast<T*>(out), s)
  if (precision == SEQDIFF_FP32) return SD_ATF(float, attention_train_fwd);
  SD_CHECK(precision == SEQDIFF_BF16 || precision == SEQDIFF_FP16, "bad precision");
  if (impl == 2) {  // the pipelined tcgen05 kernel with in-kernel dropout: what the training step runs (p_drop > 0, Lk % 4 == 0)
    if (precision == SEQDIFF_BF16) return SD_ATF(bf16, attention_pipe_dropout);
    return SD_ATF(f16, attention_pipe_dropout);
  }
  if (precision == SEQDIFF_BF16) return impl ? SD_ATF(bf16, attention_train_fwd) : SD_ATF(bf16, attention_train_fwd_tc);
  return impl ? SD_ATF(f16, attention_train_fwd) : SD_ATF(f16, attention_train_fwd_tc);
#undef SD_ATF
  SD_GUARD_END
}
int seqdiff_op_attention_train_bwd(int precision, int impl, int B, int heads, int Lq, int Lk, const void* q, int ldq, const void* k, int ldk,
                                   const void* v, int ldv, const void* dist_emb, int P, const float* key_mask, float p_drop, uint64_t seed,
                                   uint32_t site, uint32_t step, const void* dout, void* dq, void* dk, void* dv, float* dE, void* stream) {
  SD_GUARD_BEGIN
  SD_CHECK(q && k && v && key_mask && dout && dq && dk && dv, "null argument");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const DropSpec dr{p_drop, site, step, seed};
  const int Hh = heads * 64;
#define SD_ATB(T, FN) FN<T>(B, heads, Lq, Lk, static_cast<const T*>(q), ldq, static_cast<const T*>(k), ldk, static_cast<const T*>(v), ldv, \
                           static_cast<const T*>(dist_emb), P, key_mask, dr, static_cast<const T*>(dout), static_cast<T*>(dq), Hh,        \
                           static_cast<T*>(dk), Hh, static_cast<T*>(dv), Hh, dE, s)
  if (precision == SEQDIFF_FP32) return SD_ATB(float, attention_bwd);
  if (impl == 3) {  // tcgen05 backward (Lq / Lk <= 128)
    if (precision == SEQDIFF_BF16) return SD_ATB(bf16, attention_bwd_pipe);
    return SD_ATB(f16, attention_bwd_pipe);
  }
  if (precision == SEQDIFF_BF16) return impl ? SD_ATB(bf16, attention_bwd) : SD_ATB(bf16, attention_bwd_tc);
  SD_CHECK(precision == SEQDIFF_FP16, "bad precision");
  return impl ? SD_ATB(f16, attention_bwd) : SD_ATB(f16, attention_bwd_tc);
#undef SD_ATB
  SD_GUARD_END
}

int seqdiff_op_gemm_tn(int precision, int M, int N, int K, const void* At, const void* Bt, float* C, int split_k, void* stream) {
  SD_GUARD_BEGIN
  SD_CHECK(At && Bt && C, "null argument");
  SD_CHECK(precision == SEQDIFF_BF16 || precision == SEQDIFF_FP16, "the TN product exists for the 16-bit modes");
  static float* zero_bias = nullptr;  // (test entry point: one process-lifetime buffer)
  if (!zero_bias) {
    SD_CUDA(cudaMalloc(reinterpret_cast<void**>(&zero_bias), 16384 * sizeof(float)));
    SD_CUDA(cudaMemset(zero_bias, 0, 16384 * sizeof(float)));
  }
  SD_CHECK(N <= 16384, "N too large for the test entry point");
  return gemm_16_tn(M, N, K, At, Bt, precision == SEQDIFF_BF16 ? 1 : 0, zero_bias, C, static_cast<cudaStream_t>(stream), split_k);
  SD_GUARD_END
}

int seqdiff_op_layernorm(int precision, int M, int H, const float* in, const float* ln_w, const float* ln_b, float eps, float* out32, void* out16,
                         float* stats, void* stream) {
  SD_GUARD_BEGIN
  SD_CHECK(in && ln_w && ln_b && (out32 || out16) && M > 0, "bad argument");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  float2* st = reinterpret_cast<float2*>(stats);
  if (precision == SEQDIFF_FP32) return layernorm<float>(in, M, H, ln_w, ln_b, eps, out32, nullptr, st, s);
  if (precision == SEQDIFF_FP16) return layernorm<f16>(in, M, H, ln_w, ln_b, eps, out32, static_cast<f16*>(out16), st, s);
  SD_CHECK(precision == SEQDIFF_BF16, "bad precision");
  return layernorm<bf16>(in, M, H, ln_w, ln_b, eps, out32, static_cast<bf16*>(out16), st, s);
  SD_GUARD_END
}

int seqdiff_op_philox_u32(uint64_t seed, uint64_t graph_id0, uint32_t step, int B, int L, uint32_t* out, void* stream) {
  SD_GUARD_BEGIN
  SD_CHECK(out && B > 0 && L > 0, "bad argument");
  return philox_u32(seed, graph_id0, step, B, L, out, static_cast<cudaStream_t>(stream));
  SD_GUARD_END
}

}  // extern "C"
