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

int seqdiff_struct_train_step(seqdiff_model_t* m, int precision, int B, int L_lig, int L_rec, const float* timestep, const float* corrupted,
                              const float* known_noise, const float* ligand_mask, const float* receptor_seq, const float* receptor_angles,
                              const float* receptor_mask, float p_hidden, float p_attn, uint64_t seed, uint32_t step, float* grads_out,
                              double* terms_out, float* pred_out, void* stream) {
  SD_GUARD_BEGIN
  SD_CHECK(m && timestep && corrupted && known_noise && ligand_mask && receptor_seq && receptor_angles && receptor_mask && grads_out && terms_out,
           "null argument");
  StructTrainArgs a{};
  a.precision = precision; a.B = B; a.Ll = L_lig; a.Lr = L_rec;
  a.t = timestep; a.corrupted = corrupted; a.known_noise = known_noise; a.lig_mask = ligand_mask;
  a.rec_seq = receptor_seq; a.rec_angle = receptor_angles; a.rec_mask = receptor_mask;
  a.p_hidden = p_hidden; a.p_attn = p_attn; a.seed = seed; a.step = step;
  a.grads = grads_out; a.terms = terms_out; a.pred_out = pred_out;
  return m->impl.struct_train_step(a, static_cast<cudaStream_t>(stream));
  SD_GUARD_END
}

int seqdiff_struct_loss_terms(int N, int F, const float* pred, const float* known_noise, const float* ligand_mask, double* terms, void* stream) {
  SD_GUARD_BEGIN
  SD_CHECK(pred && known_noise && ligand_mask && terms, "null argument");
  return angle_loss_terms(N, F, pred, known_noise, ligand_mask, terms, static_cast<cudaStream_t>(stream));
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

int seqdiff_score_multi(seqdiff_model_t* m, int precision, int P, int K, int L_lig, int L_rec, int T, const float* q_tables_steps,
                        const float* x0, const float* ligand_angle, const float* ligand_mask, const float* receptor_seq,
                        const float* receptor_angle, const float* receptor_mask, const float* noise_E_steps, uint64_t seed, uint64_t graph_id0,
                        int flags, double* terms_out, void* stream) {
  SD_GUARD_BEGIN
  SD_CHECK(m && q_tables_steps && x0 && ligand_angle && ligand_mask && receptor_seq && receptor_angle && receptor_mask && terms_out,
           "null argument");
  SD_CHECK(P >= 1 && K >= 1 && T >= 1, "need at least one pocket, one sample per pocket and one step");
  SD_CHECK(L_lig > 0 && L_rec > 0 && static_cast<int64_t>(P) * K * (L_lig > L_rec ? L_lig : L_rec) <= INT32_MAX,
           "pockets x samples x length overflows the row counts");
  SD_CHECK((flags & ~1) == 0, "unknown scoring flag");
  SD_CHECK(m->impl.cfg.feature_size == SEQDIFF_NUM_CLASSES, "scoring needs feature_size == 20");
  return m->impl.score(precision, P, K, L_lig, L_rec, T, q_tables_steps, x0, ligand_angle, ligand_mask, receptor_seq, receptor_angle,
                       receptor_mask, noise_E_steps, seed, graph_id0, terms_out, static_cast<cudaStream_t>(stream), flags);
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
  return m->impl.struct_sample(precision, B, 1, L_lig, L_rec, T, coef_steps, x_T, ligand_mask, receptor_seq, receptor_angles, receptor_mask,
                               noise_steps, seed, graph_id0, steps_out, final_out, static_cast<cudaStream_t>(stream), 0);
  SD_GUARD_END
}

int seqdiff_struct_sample_ex(seqdiff_model_t* m, int precision, int B, int L_lig, int L_rec, int T, const float* coef_steps, const float* x_T,
                             const float* ligand_mask, const float* receptor_seq, const float* receptor_angles, const float* receptor_mask,
                             const float* noise_steps, uint64_t seed, uint64_t graph_id0, int flags, float* steps_out, float* final_out,
                             void* stream) {
  return seqdiff_struct_sample_multi(m, precision, B, 1, L_lig, L_rec, T, coef_steps, x_T, ligand_mask, receptor_seq, receptor_angles,
                                     receptor_mask, noise_steps, seed, graph_id0, flags, steps_out, final_out, stream);
}

int seqdiff_struct_sample_multi(seqdiff_model_t* m, int precision, int P, int K, int L_lig, int L_rec, int T, const float* coef_steps,
                                const float* x_T, const float* ligand_mask, const float* receptor_seq, const float* receptor_angles,
                                const float* receptor_mask, const float* noise_steps, uint64_t seed, uint64_t graph_id0, int flags,
                                float* steps_out, float* final_out, void* stream) {
  SD_GUARD_BEGIN
  SD_CHECK(m && coef_steps && x_T && ligand_mask && receptor_seq && receptor_angles && receptor_mask && final_out, "null argument");
  SD_CHECK(P >= 1 && K >= 1, "need at least one pocket and one sample per pocket");
  SD_CHECK(L_lig > 0 && L_rec > 0 && static_cast<int64_t>(P) * K * (L_lig > L_rec ? L_lig : L_rec) <= INT32_MAX,
           "pockets x samples x length overflows the row counts");
  SD_CHECK((flags & ~1) == 0, "unknown sampling flag");
  return m->impl.struct_sample(precision, P, K, L_lig, L_rec, T, coef_steps, x_T, ligand_mask, receptor_seq, receptor_angles, receptor_mask,
                               noise_steps, seed, graph_id0, steps_out, final_out, static_cast<cudaStream_t>(stream), flags);
  SD_GUARD_END
}

int seqdiff_struct_score_multi(seqdiff_model_t* m, int precision, int P, int K, int L_lig, int L_rec, int T, const float* qs_steps,
                               const float* x0, const float* ligand_mask, const float* receptor_seq, const float* receptor_angles,
                               const float* receptor_mask, const float* noise_steps, uint64_t seed, uint64_t graph_id0, int flags,
                               double* terms_out, void* stream) {
  SD_GUARD_BEGIN
  SD_CHECK(m && qs_steps && x0 && ligand_mask && receptor_seq && receptor_angles && receptor_mask && terms_out, "null argument");
  SD_CHECK(P >= 1 && K >= 1 && T >= 1, "need at least one pocket, one backbone per pocket and one step");
  SD_CHECK(L_lig > 0 && L_rec > 0 && static_cast<int64_t>(P) * K * (L_lig > L_rec ? L_lig : L_rec) <= INT32_MAX,
           "pockets x backbones x length overflows the row counts");
  SD_CHECK(static_cast<int64_t>(P) * K <= 65535, "more than 65535 backbones in one call (the step kernels put one graph per grid row)");
  SD_CHECK((flags & ~1) == 0, "unknown scoring flag");
  SD_CHECK(m->impl.arch == kArchStructure, "handle holds a sequence model: use seqdiff_score_multi");
  return m->impl.struct_score(precision, P, K, L_lig, L_rec, T, qs_steps, x0, ligand_mask, receptor_seq, receptor_angles, receptor_mask,
                              noise_steps, seed, graph_id0, terms_out, static_cast<cudaStream_t>(stream), flags);
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

int seqdiff_op_gemm_ex(int precision, int M, int N, int K, const void* A, const void* W, const float* bias, const float* resid, const float* ln_stats,
                       const float* ln_g, const float* ln_b, int epilogue, int out_f32, int split_k, void* C, void* stream) {
  SD_GUARD_BEGIN
  SD_CHECK(A && W && bias && C, "null argument");
  const int force_bn = ((precision >> 8) & 0xfff) | (((precision >> 20) & 1) << 16);
  const int mode = precision & 0xff;
  SD_CHECK(mode == SEQDIFF_BF16 || mode == SEQDIFF_FP16, "the tcgen05 GEMM forms exist for the 16-bit modes");
  const int fmt = mode == SEQDIFF_FP16 ? 0 : 1;
  const LnResid ln{reinterpret_cast<const float2*>(ln_stats), ln_g, ln_b};
  return gemm_16(M, N, K, A, fmt, W, fmt, bias, resid, epilogue, C, out_f32 ? 2 : fmt, static_cast<cudaStream_t>(stream), force_bn,
                 ln_stats ? &ln : nullptr, split_k);
  SD_GUARD_END
}

int seqdiff_op_attention_packed(int precision, int B, int heads, int Lq, int Lk, const void* q, int ldq, const void* k, int ldk, const void* v,
                                int ldv, const void* dist_emb, int P, const float* key_mask, int Lk_mask, const int* q_off, const int* k_off,
                                const int* q_len, int q_rows, int k_rows, int kv_div, void* out, void* stream) {
  SD_GUARD_BEGIN
  SD_CHECK(q && k && v && key_mask && out, "null argument");
  SD_CHECK(q_off || (!k_off && !q_len && Lk_mask == Lk), "padded form (q_off NULL): no k_off / q_len, and the key-mask pitch is Lk");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const AttnPack pk{q_off, k_off, q_len, q_rows, k_rows, Lk_mask};
  const AttnPack* pack = q_off ? &pk : nullptr;
  if (precision == SEQDIFF_FP32)
    return attention<float>(B, heads, Lq, Lk, static_cast<const float*>(q), ldq, static_cast<const float*>(k), ldk, static_cast<const float*>(v),
                            ldv, static_cast<const float*>(dist_emb), P, key_mask, static_cast<float*>(out), s, pack, kv_div);
  if (precision == SEQDIFF_FP16)
    return attention<f16>(B, heads, Lq, Lk, static_cast<const f16*>(q), ldq, static_cast<const f16*>(k), ldk, static_cast<const f16*>(v), ldv,
                          static_cast<const f16*>(dist_emb), P, key_mask, static_cast<f16*>(out), s, pack, kv_div);
  SD_CHECK(precision == SEQDIFF_BF16, "bad precision");
  return attention<bf16>(B, heads, Lq, Lk, static_cast<const bf16*>(q), ldq, static_cast<const bf16*>(k), ldk, static_cast<const bf16*>(v), ldv,
                         static_cast<const bf16*>(dist_emb), P, key_mask, static_cast<bf16*>(out), s, pack, kv_div);
  SD_GUARD_END
}

// ---- training-step rowwise / elementwise kernels, operator level (train_kernels.cu, decode_loss.cu) ----------------------------------------
// Thin: every form a kernel does not implement is rejected here, before anything reaches the device; the launchers are called as the training
// step calls them.  Row-vector operands are read and written 16 bytes at a time, so their pointers must be 16 B aligned; the accumulated
// parameter gradients may sit at any float offset (the flushes pick 128-bit or scalar atomics from the alignment).
}  // extern "C"
namespace {
bool is_a16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }
bool rowwise_h(int H) { return H == 256 || H == 512 || H == 768 || H == 1024; }
bool mode_ok(int precision) { return precision == SEQDIFF_FP32 || precision == SEQDIFF_BF16 || precision == SEQDIFF_FP16; }
}  // namespace
extern "C" {

int seqdiff_op_dropout_add_layernorm(int precision, int M, int H, float* d, const float* resid, const float* ln_w, const float* ln_b, float eps,
                                     float p, uint64_t seed, uint32_t site, uint32_t step, float* out32, void* out16, uint8_t* keep_bits,
                                     void* stream) {
  SD_GUARD_BEGIN
  SD_CHECK(d && resid && ln_w && ln_b, "null argument");
  SD_CHECK(mode_ok(precision) && M > 0 && rowwise_h(H), "precision, M > 0 and H in {256, 512, 768, 1024}");
  SD_CHECK(precision != SEQDIFF_FP32 || !out16, "FP32 has no 16-bit output");
  SD_CHECK(is_a16(d) && is_a16(resid) && is_a16(ln_w) && is_a16(ln_b) && is_a16(out32) && is_a16(out16), "row pointers must be 16 B aligned");
  const DropSpec dr{p, site, step, seed};
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (precision == SEQDIFF_FP32) return dropout_add_layernorm<float>(d, resid, dr, M, H, ln_w, ln_b, eps, out32, nullptr, keep_bits, s);
  if (precision == SEQDIFF_BF16)
    return dropout_add_layernorm<bf16>(d, resid, dr, M, H, ln_w, ln_b, eps, out32, static_cast<bf16*>(out16), keep_bits, s);
  return dropout_add_layernorm<f16>(d, resid, dr, M, H, ln_w, ln_b, eps, out32, static_cast<f16*>(out16), keep_bits, s);
  SD_GUARD_END
}

int seqdiff_op_layernorm_bwd(int precision, int M, int H, const float* dh, const float* o, const float* gamma, float eps, float* d_o, float* dgamma,
                             float* dbeta, float p, uint64_t seed, uint32_t site, uint32_t step, const uint8_t* keep_bits, void* g16, float* dbias,
                             void* stream) {
  SD_GUARD_BEGIN
  SD_CHECK(dh && o && gamma && d_o && dgamma && dbeta, "null argument");
  SD_CHECK(mode_ok(precision) && M > 0 && rowwise_h(H), "precision, M > 0 and H in {256, 512, 768, 1024}");
  SD_CHECK(is_a16(dh) && is_a16(o) && is_a16(gamma) && is_a16(d_o) && is_a16(g16), "row pointers must be 16 B aligned");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (precision == SEQDIFF_FP32) {
    SD_CHECK(!g16 && !dbias && !keep_bits && p == 0.f, "FP32: the plain LayerNorm backward (no 16-bit operand, bias gradient or dropout)");
    return layernorm_bwd(dh, o, M, H, gamma, eps, d_o, dgamma, dbeta, s);
  }
  SD_CHECK(g16 && dbias, "16-bit modes: the 16-bit dY operand and the bias gradient are required");
  const DropSpec dr{p, site, step, seed};
  if (precision == SEQDIFF_BF16)
    return layernorm_bwd_cast<bf16>(dh, o, M, H, gamma, eps, d_o, dgamma, dbeta, dr, keep_bits, static_cast<bf16*>(g16), dbias, s);
  return layernorm_bwd_cast<f16>(dh, o, M, H, gamma, eps, d_o, dgamma, dbeta, dr, keep_bits, static_cast<f16*>(g16), dbias, s);
  SD_GUARD_END
}

int seqdiff_op_ln_modulate_bwd(int precision, int M, int H, const float* dout, const float* in, int affine_first, const float* lnw, const float* lnb,
                               float eps1, const void* mod, int mod_div, int chunk0, float* din, float* sum_out, void* dmodT, float* dmod32,
                               float* dgamma, float* dbeta, void* stream) {
  SD_GUARD_BEGIN
  SD_CHECK(dout && in && mod && din, "null argument");
  SD_CHECK(mode_ok(precision) && M > 0 && rowwise_h(H), "precision, M > 0 and H in {256, 512, 768, 1024}");
  SD_CHECK(!affine_first || (lnw && lnb && dgamma && dbeta), "affine_first needs the LayerNorm affine and its gradients");
  SD_CHECK((dmodT != nullptr) != (dmod32 != nullptr), "exactly one of dmodT / dmod32");
  SD_CHECK(mod_div >= 1 && (!dmodT || mod_div == 1), "mod_div >= 1; per-token rows (dmodT) need mod_div == 1");
  SD_CHECK(chunk0 >= 0 && chunk0 <= 3, "chunk0: the (shift, scale, gate) triple starts at chunk 0 .. 3 of the 6H row");
  SD_CHECK(is_a16(dout) && is_a16(in) && is_a16(lnw) && is_a16(lnb) && is_a16(mod) && is_a16(din) && is_a16(sum_out) && is_a16(dmodT),
           "row pointers must be 16 B aligned");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
#define SD_LMB(T) ln_modulate_bwd<T>(dout, in, M, H, affine_first != 0, lnw, lnb, eps1, static_cast<const T*>(mod), mod_div, chunk0, din, sum_out, \
                                     static_cast<T*>(dmodT), dmod32, dgamma, dbeta, s)
  if (precision == SEQDIFF_FP32) return SD_LMB(float);
  if (precision == SEQDIFF_BF16) return SD_LMB(bf16);
  return SD_LMB(f16);
#undef SD_LMB
  SD_GUARD_END
}

int seqdiff_op_embed_bwd(int M, int fin, int H, const float* dout, const float* x, const float* Wt, const float* b, const float* gamma, float eps,
                         float p, uint64_t seed, uint32_t site, uint32_t step, float* dW, float* db, float* dgamma, float* dbeta, void* stream) {
  SD_GUARD_BEGIN
  SD_CHECK(dout && x && Wt && b && gamma && dW && db && dgamma && dbeta, "null argument");
  SD_CHECK(M > 0 && rowwise_h(H) && fin >= 1 && fin <= 32, "M > 0, H in {256, 512, 768, 1024} and fin in [1, 32]");
  SD_CHECK(is_a16(dout) && is_a16(Wt) && is_a16(b) && is_a16(gamma), "row pointers must be 16 B aligned");
  return embed_bwd(dout, x, M, fin, H, Wt, b, gamma, eps, DropSpec{p, site, step, seed}, dW, db, dgamma, dbeta, static_cast<cudaStream_t>(stream));
  SD_GUARD_END
}

int seqdiff_op_predictor_tail_bwd(int precision, int M, int H, int F, const float* dlogits, const void* y, const float* gamma, const float* beta,
                                  float eps, const float* W2, float* dy, float* dW2, float* db2, float* dgamma, float* dbeta, void* stream) {
  SD_GUARD_BEGIN
  SD_CHECK(dlogits && y && gamma && beta && W2 && dy && dW2 && db2 && dgamma && dbeta, "null argument");
  SD_CHECK(mode_ok(precision) && M > 0 && rowwise_h(H) && (F == 8 || F == 20), "precision, M > 0, H in {256, 512, 768, 1024} and F in {8, 20}");
  SD_CHECK(is_a16(y) && is_a16(gamma) && is_a16(beta) && is_a16(W2) && is_a16(dy), "row pointers must be 16 B aligned");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
#define SD_PTB(T) predictor_tail_bwd<T>(dlogits, static_cast<const T*>(y), M, H, gamma, beta, eps, W2, F, dy, dW2, db2, dgamma, dbeta, s)
  if (precision == SEQDIFF_FP32) return SD_PTB(float);
  if (precision == SEQDIFF_BF16) return SD_PTB(bf16);
  return SD_PTB(f16);
#undef SD_PTB
  SD_GUARD_END
}

int seqdiff_op_train_elementwise(int op, int precision, int64_t n, int kind, const void* in, const void* aux, float p, uint64_t seed, uint32_t site,
                                 uint32_t step, void* out, void* stream) {
  SD_GUARD_BEGIN
  SD_CHECK(out && (in || op == 4), "null argument");
  SD_CHECK(mode_ok(precision) && n > 0 && n % 8 == 0, "precision and n > 0, n % 8 == 0");
  SD_CHECK(op >= 0 && op <= 4, "op: 0 act_fwd, 1 act_bwd, 2 act_bwd (fp32 gradient), 3 grad_cast, 4 dropout_add");
  SD_CHECK(op > 2 || kind == 1 || kind == 2, "activation kind: 1 erf-GELU, 2 SiLU");
  SD_CHECK(op == 0 || op == 3 || op == 4 || aux, "act_bwd needs z");
  SD_CHECK(op != 4 || precision == SEQDIFF_FP32, "dropout_add is fp32");
  SD_CHECK(is_a16(in) && is_a16(aux) && is_a16(out), "pointers must be 16 B aligned");
  const DropSpec dr{p, site, step, seed};
  const size_t m = static_cast<size_t>(n);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (op == 4) return dropout_add(static_cast<float*>(out), static_cast<const float*>(in), m, dr, s);
#define SD_EW(T)                                                                                                                          \
  switch (op) {                                                                                                                           \
    case 0: return act_fwd<T>(static_cast<const T*>(in), m, kind, dr, static_cast<T*>(out), s);                                          \
    case 1: return act_bwd<T, T>(static_cast<const T*>(in), static_cast<const T*>(aux), m, kind, dr, static_cast<T*>(out), s);           \
    case 2: return act_bwd<T, float>(static_cast<const float*>(in), static_cast<const T*>(aux), m, kind, dr, static_cast<T*>(out), s);   \
    default: return grad_cast<T>(static_cast<const float*>(in), m, dr, static_cast<T*>(out), s);                                        \
  }
  if (precision == SEQDIFF_FP32) { SD_EW(float) }
  if (precision == SEQDIFF_BF16) { SD_EW(bf16) }
  SD_EW(f16)
#undef SD_EW
  SD_GUARD_END
}

int seqdiff_op_transpose_colsum(int precision, int rows, int cols, const void* in, void* out, int pitch, float* colsum, void* stream) {
  SD_GUARD_BEGIN
  SD_CHECK(in && (out || colsum), "null argument");
  SD_CHECK(mode_ok(precision) && rows > 0 && cols > 0, "precision, rows > 0 and cols > 0");
  SD_CHECK(pitch == 0 || (pitch >= rows && pitch - rows < 64), "pitch: 0 (= rows) or rows rounded up by less than one 64-row tile");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (precision == SEQDIFF_FP32)
    return transpose_colsum<float>(static_cast<const float*>(in), rows, cols, static_cast<float*>(out), colsum, s, pitch);
  if (precision == SEQDIFF_BF16) return transpose_colsum<bf16>(static_cast<const bf16*>(in), rows, cols, static_cast<bf16*>(out), colsum, s, pitch);
  return transpose_colsum<f16>(static_cast<const f16*>(in), rows, cols, static_cast<f16*>(out), colsum, s, pitch);
  SD_GUARD_END
}

int seqdiff_op_colsum_add(int precision, int rows, int cols, const void* in, float* colsum, void* stream) {
  SD_GUARD_BEGIN
  SD_CHECK(in && colsum, "null argument");
  SD_CHECK(precision == SEQDIFF_BF16 || precision == SEQDIFF_FP16, "the column sum exists for the 16-bit modes");
  SD_CHECK(rows > 0 && cols > 0 && cols % 8 == 0 && is_a16(in), "rows > 0, cols a multiple of 8, 16 B aligned input");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (precision == SEQDIFF_BF16) return colsum_add<bf16>(static_cast<const bf16*>(in), rows, cols, colsum, s);
  return colsum_add<f16>(static_cast<const f16*>(in), rows, cols, colsum, s);
  SD_GUARD_END
}

int seqdiff_op_loss_bwd(int N, const float* logits, const float* x0, const float* x_t, const double* terms, float* dlogits, void* stream) {
  SD_GUARD_BEGIN
  SD_CHECK(logits && x0 && x_t && terms && dlogits, "null argument");
  SD_CHECK(is_a16(logits) && is_a16(x0) && is_a16(x_t) && is_a16(dlogits), "row pointers must be 16 B aligned");
  return loss_bwd(N, logits, x0, x_t, terms, dlogits, static_cast<cudaStream_t>(stream));
  SD_GUARD_END
}

int seqdiff_op_angle_loss_bwd(int N, int F, const float* pred, const float* noise, const float* mask, const double* terms, float* dpred,
                              void* stream) {
  SD_GUARD_BEGIN
  SD_CHECK(pred && noise && mask && terms && dpred, "null argument");
  return angle_loss_bwd(N, F, pred, noise, mask, terms, dpred, static_cast<cudaStream_t>(stream));
  SD_GUARD_END
}

}  // extern "C"
