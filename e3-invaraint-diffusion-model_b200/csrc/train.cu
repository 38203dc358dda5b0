// train.cu -- the training step of the sequence denoiser (BASELINE configs[3]): forward with dropout + loss + full backward into one
// flat fp32 gradient buffer, and the clip + AdamW update.  Replaces, for one optimizer step, what the reference gets from autograd
// over PeptideDiff.training_step / get_loss (sequence_model/model.py:313-367), torch.optim.AdamW (model.py:420-422) and Lightning's
// gradient_clip_val (train_model.py:95).  The data-parallel gradient all-reduce happens BETWEEN the two entry points, on the
// caller's flat buffer (train.py: torch.distributed over NCCL) -- the library itself never communicates.
//
// Forward.  Same kernels as inference (tcgen05 GEMMs, rowwise kernels) in the plain post-LN flow, with every tensor the backward
// needs kept on a tape in the training workspace: 16-bit operands of each GEMM, fp32 pre-LayerNorm tensors, pre-activation values.
// LayerNorm statistics, softmax probabilities and dropout masks are NOT stored: they are recomputed / regenerated.
//
// Backward of a Linear y = x W^T + b, all three products on the tcgen05 GEMM (C = A B^T with both operands K-major):
//   dx = dy W          = gemm(A = dy [M,N],      B = W^T [K,N])   -- W^T: transposed operand copy made once per optimizer step
//   dW = dy^T x        = gemm(A = dy^T [N,M],    B = x^T [K,M])   -- 16-bit transposes of dy and x (one HBM round trip each)
//   db = column sums of dy (fused into the transpose of dy)
// Residual-stream gradients stay fp32; a gradient becomes 16-bit only as a GEMM operand.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <type_traits>

#include "model.cuh"

namespace seqdiff {

template <typename T> struct TFmt;
template <> struct TFmt<f16> { static constexpr int v = 0; };
template <> struct TFmt<bf16> { static constexpr int v = 1; };
template <> struct TFmt<float> { static constexpr int v = -1; };

static size_t al256(size_t b) { return (b + 255) & ~static_cast<size_t>(255); }
struct Arena {
  uint8_t* p;
  uint8_t* end;
  cudaStream_t gs;    // debug build: stream the guard bands are filled on (common.cuh: SEQDIFF_DEBUG_BOUNDS)
  const void* owner;
  bool ok = true;
  Arena(uint8_t* base, uint8_t* e, cudaStream_t s) : p(base), end(e), gs(s), owner(base) { debug_guard_begin(owner); }
  template <typename T> T* take(size_t n) {
    T* r = reinterpret_cast<T*>(p);
    p += al256(n * sizeof(T));
    if (kGuardBytes && p + kGuardBytes <= end) {
      debug_guard_add(owner, p, gs);
      p += kGuardBytes;
    }
    if (p > end) ok = false;
    return r;
  }
};

// C[M,N] = A[M,K] B[N,K]^T + bias (+ resid); out_f32: fp32 C (always in fp32 mode)
template <typename T>
static int gemm_any(int M, int N, int K, const T* A, const void* Bw, const float* bias, const float* resid, void* C, bool out_f32, cudaStream_t s,
                    int split_k = 1) {
  if constexpr (std::is_same<T, float>::value) {
    return gemm_f32(M, N, K, A, static_cast<const float*>(Bw), bias, resid, 0, static_cast<float*>(C), s);
  } else {
    return gemm_16(M, N, K, A, TFmt<T>::v, Bw, TFmt<T>::v, bias, resid, 0, C, (out_f32 || resid) ? 2 : TFmt<T>::v, s, 0, nullptr, split_k);
  }
}
template <typename T> static const void* wsel(const Wt& w) {
  if constexpr (std::is_same<T, float>::value) return w.f;
  else if constexpr (std::is_same<T, bf16>::value) return w.h;
  else return w.g;
}

// v = dropout(v) [+ te[row / L]] -> out32 (in place) and the operand copy: BertEmbeddings.dropout (model.py:116) when p > 0
template <typename T>
__global__ void __launch_bounds__(256) embed_post_kernel(float* __restrict__ v, const float* __restrict__ te, int L, int H, size_t n8, DropSpec dr,
                                                         float* __restrict__ out32, T* __restrict__ outT) {
  pdl_wait();
  for (size_t i = static_cast<size_t>(blockIdx.x) * 256 + threadIdx.x; i < n8; i += static_cast<size_t>(gridDim.x) * 256) {
    float x[8], keep[8];
    load8<float>(v + 8 * i, x);
    drop_scales8(dr, 8 * i, keep);
#pragma unroll
    for (int j = 0; j < 8; ++j) x[j] *= keep[j];
    if (te) {
      const size_t row = (8 * i) / H, col = (8 * i) % H;
      float t8[8];
      load8<float>(te + (row / L) * H + col, t8);
#pragma unroll
      for (int j = 0; j < 8; ++j) x[j] += t8[j];
    }
    if (out32) store8<float>(out32 + 8 * i, x);
    if (outT) store8<T>(outT + 8 * i, x);
  }
}
template <typename T>
static int embed_post(float* v, const float* te, int L, int H, size_t n, DropSpec dr, float* out32, T* outT, cudaStream_t s) {
  const size_t n8 = n / 8;
  const int grid = static_cast<int>(n8 / 256 + 1 < 2048 ? n8 / 256 + 1 : 2048);
  SD_CUDA(launch_k(embed_post_kernel<T>, dim3(grid), dim3(256), 0, s, v, te, L, H, n8, dr, out32, std::is_same<T, float>::value ? nullptr : outT));
  SD_LAUNCHED("embed_post", s);
  return SEQDIFF_OK;
}
__global__ void concat_masks_kernel(float* dst, const float* a, int na, const float* b, int nb) {
  pdl_wait();
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < na + nb; i += gridDim.x * blockDim.x) dst[i] = i < na ? a[i] : b[i - na];
}

// =====================================================================================================
// parameter table
// =====================================================================================================
int Model::build_slots() {
  if (!slots.empty()) return SEQDIFF_OK;
  const int NL = cfg.num_hidden_layers;
  int64_t off = 0;
  bool missing = false;
  auto add = [&](const std::string& n) {
    auto it = raw.find(n);
    if (it == raw.end() || !it->second.ptr) { missing = true; return; }
    ParamSlot ps;
    ps.name = n;
    ps.w = it->second.ptr;
    ps.numel = it->second.numel;
    ps.off = off;
    off += (ps.numel + 3) & ~static_cast<int64_t>(3);  // 16 B aligned starts (vectorised optimizer / reductions)
    slot_of[n] = static_cast<int>(slots.size());
    slots.push_back(ps);
  };
  auto attn = [&](const std::string& p, bool rel) {
    for (const char* n : {"query", "key", "value"}) add(p + ".self." + n + ".weight");
    for (const char* n : {"query", "key", "value"}) add(p + ".self." + n + ".bias");
    if (rel && cfg.relative_key) add(p + ".self.distance_embedding.weight");
    add(p + ".output.dense.weight");
    add(p + ".output.dense.bias");
    add(p + ".output.LayerNorm.weight");
    add(p + ".output.LayerNorm.bias");
  };
  auto emb = [&](const std::string& e) {
    for (const char* t : {".linear.weight", ".linear.bias", ".LayerNorm.weight", ".LayerNorm.bias"}) add(e + t);
  };
  // The flat index space follows the FORWARD order of the network, so the backward pass finishes it from the end towards the start
  // and the data-parallel all-reduce can start on the tail buckets while the head of the buffer is still being computed
  // (grad_bucket_bounds, bucket_events).  receptor_feature_emb: dead weight, no gradient (quirk Q1).
  auto se_block = [&](const std::string& p) {
    add(p + ".adaLN_modulation.0.weight");
    add(p + ".adaLN_modulation.0.bias");
    add(p + ".adaLN_modulation.2.weight");
    add(p + ".adaLN_modulation.2.bias");
    attn(p + ".attn", true);
    add(p + ".mlp.0.weight");
    add(p + ".mlp.0.bias");
    add(p + ".mlp.3.weight");
    add(p + ".mlp.3.bias");
  };
  auto ffn = [&](const std::string& p) {
    add(p + ".intermediate.dense.weight");
    add(p + ".intermediate.dense.bias");
    add(p + ".output.dense.weight");
    add(p + ".output.dense.bias");
    add(p + ".output.LayerNorm.weight");
    add(p + ".output.LayerNorm.bias");
  };
  // cross-attention K | V of every layer: contiguous in the order of the fused [layers * 2H, H] projection
  auto cross_kv = [&]() {
    for (int i = 0; i < NL; ++i)
      for (const char* n : {"key", "value"}) add("decoder.layer." + std::to_string(i) + ".crossattention.self." + n + ".weight");
    for (int i = 0; i < NL; ++i)
      for (const char* n : {"key", "value"}) add("decoder.layer." + std::to_string(i) + ".crossattention.self." + n + ".bias");
  };
  auto decoder = [&]() {
    for (int i = 0; i < NL; ++i) {
      const std::string p = "decoder.layer." + std::to_string(i);
      if (i == NL / 2 && i > 0) grad_bucket_bounds.push_back(off);  // next bucket: the second half of the decoder layers
      attn(p + ".attention", true);
      add(p + ".crossattention.self.query.weight");
      add(p + ".crossattention.self.query.bias");
      add(p + ".crossattention.output.dense.weight");
      add(p + ".crossattention.output.dense.bias");
      add(p + ".crossattention.output.LayerNorm.weight");
      add(p + ".crossattention.output.LayerNorm.bias");
      ffn(p);
    }
  };
  auto head = [&](const std::string& h) {
    for (const char* t : {"dense1.weight", "dense1.bias", "layer_norm.weight", "layer_norm.bias", "dense2.weight", "dense2.bias"}) add(h + "." + t);
  };
  grad_bucket_bounds.clear();
  grad_bucket_bounds.push_back(0);
  if (arch == kArchSequence) {
    for (const char* e : {"ligand_seq_embedding", "ligand_angle_embedding", "receptor_seq_embedding", "receptor_angle_embedding"}) emb(e);
    se_block("ligand_feature_emb");       // bucket 0: the four embeddings + ligand_feature_emb (finished last)
    grad_bucket_bounds.push_back(off);    // bucket 1: fused cross K | V + the first half of the decoder layers
    cross_kv();
    decoder();                            // (bucket 2: the second half of the decoder layers)
    grad_bucket_bounds.push_back(off);    // last bucket: decoder_normalize + the predictor head (finished first)
    se_block("decoder_normalize");
    head("amino_acid_predictor");
  } else {
    // structure model.  Buckets, finished from the last: [decoder second half + head], [fused cross K | V + ligand_angle_emb +
    // timestep_emb + decoder first half] (final once the encoder-output gradient GEMM has run), [encoder second half], [receptor
    // embeddings + receptor_emb + encoder first half].  The first two are all-reduced under the encoder backward.
    emb("receptor_seq_emb");
    emb("receptor_angle_emb");
    se_block("receptor_emb");
    for (int i = 0; i < NL; ++i) {
      const std::string p = "encoder.layer." + std::to_string(i);
      if (i == NL / 2 && i > 0) grad_bucket_bounds.push_back(off);
      attn(p + ".attention", true);
      ffn(p);
    }
    grad_bucket_bounds.push_back(off);
    cross_kv();
    emb("ligand_angle_emb");
    se_block("timestep_emb");
    decoder();
    head("angles_predictor");
  }
  grad_bucket_bounds.push_back(off);
  if (missing) {
    slots.clear();
    slot_of.clear();
    set_error("training: every tensor must be set before the parameter table is built");
    return SEQDIFF_ERR_STATE;
  }
  train_total = off;
  // device tables for the optimizer
  std::vector<float*> hw(slots.size());
  std::vector<int64_t> ho(slots.size() + 1);
  for (size_t i = 0; i < slots.size(); ++i) { hw[i] = slots[i].w; ho[i] = slots[i].off; }
  ho[slots.size()] = off;
  d_slot_w = static_cast<float**>(dalloc(hw.size() * sizeof(float*)));
  d_slot_off = static_cast<int64_t*>(dalloc(ho.size() * sizeof(int64_t)));
  d_opt_scratch = static_cast<double*>(dalloc((2 * 160 + 16) * sizeof(double) * 2));
  d_zero_bias = static_cast<float*>(dalloc(16384 * sizeof(float)));
  SD_CHECK(d_slot_w && d_slot_off && d_opt_scratch && d_zero_bias, "cudaMalloc failed");
  SD_CUDA(cudaMemcpy(d_slot_w, hw.data(), hw.size() * sizeof(float*), cudaMemcpyHostToDevice));
  SD_CUDA(cudaMemcpy(d_slot_off, ho.data(), ho.size() * sizeof(int64_t), cudaMemcpyHostToDevice));
  SD_CUDA(cudaMemset(d_opt_scratch, 0, (2 * 160 + 16) * sizeof(double) * 2));
  SD_CUDA(cudaMemset(d_zero_bias, 0, 16384 * sizeof(float)));
  return SEQDIFF_OK;
}

int64_t Model::train_param_count() {
  if (build_slots() != SEQDIFF_OK) return -1;
  return train_total;
}

int Model::get_tensor(const char* name, float* out, int64_t numel, cudaStream_t s) {
  auto it = raw.find(name);
  if (it == raw.end()) {
    set_error(std::string("unknown tensor name: ") + name);
    return SEQDIFF_ERR_STATE;
  }
  SD_CHECK(it->second.numel == numel, "size mismatch");
  SD_CHECK(it->second.ptr != nullptr, "tensor is not stored in the handle (dead weight)");
  SD_CUDA(cudaMemcpyAsync(out, it->second.ptr, static_cast<size_t>(numel) * sizeof(float), cudaMemcpyDefault, s));
  return SEQDIFF_OK;
}

int Model::adamw(const float* grads, float* m, float* v, float grad_scale, float max_norm, float lr, float beta1, float beta2, float eps, float wd,
                 int step, float* norm_out, cudaStream_t s) {
  SD_CHECK(finalized, "model not finalised");
  SD_CUDA(cudaSetDevice(device));
  SD_TRY(build_slots());
  SD_TRY(adamw_step(d_slot_w, d_slot_off, static_cast<int>(slots.size()), static_cast<size_t>(train_total), grads, m, v, grad_scale, max_norm, lr,
                    beta1, beta2, eps, wd, step, d_opt_scratch, norm_out, s));
  // the masters changed: refresh the fused / 16-bit / transposed operand copies in place (same buffers, same stream)
  repack_reuse = true;
  const int rc = finalize(s);
  repack_reuse = false;
  return rc;
}

// =====================================================================================================
// the per-sublayer code of a training step, shared by the sequence and the structure model
// =====================================================================================================
template <typename T> struct Act2 {  // residual-stream tensor: fp32 master + operand copy (the same buffer in fp32 mode)
  float* s = nullptr;
  T* t = nullptr;
  T* t_out() const { return std::is_same<T, float>::value ? nullptr : t; }
};
template <typename T> static Act2<T> take_act2(Arena& a, size_t n) {
  Act2<T> r;
  r.s = a.take<float>(n);
  if constexpr (std::is_same<T, float>::value) r.t = r.s;
  else r.t = a.take<T>(n);
  return r;
}

template <typename T> struct SETape {
  const SEW* w;
  std::string prefix;
  int M, Mc, mod_div;
  Act2<T> x, x1, out;
  const T* c;
  T *u_pre, *u, *mod, *qkv, *ctx, *m1_pre, *m1;
  float *o, *m2;
  std::vector<Segment> segs;
  std::vector<uint32_t*> keep;  // per segment: the attention dropout mask as bits (forward -> backward), or NULL
  DropSpec d_attn, d_o, d_m1, d_m2;
};
// one post-LN BERT layer: self-attention [-> cross-attention] -> FFN (the cross members stay unused in an encoder layer)
template <typename T> struct LayerTape {
  Act2<T> h, h1, h2, h3;
  T *qkv, *ctx, *cq, *ctx2, *f_pre, *f;
  float *o1, *o2, *o3;
  uint32_t *keep_self = nullptr, *keep_cross = nullptr;
  uint8_t *kb1 = nullptr, *kb2 = nullptr, *kb3 = nullptr;  // hidden-dropout masks of the three post-LN sublayers as bits (forward -> backward)
  DropSpec d_attn, d_o1, d_cattn, d_o2, d_o3;
};
// what a layer's cross-attention reads: query graph b attends to rows [b * Lk, (b + 1) * Lk) of the fused K | V block (row pitch ld)
template <typename T> struct CrossKV {
  int Lk, ld;
  const T* kv;     // this layer's K columns; V follows at + H
  T* dkv;          // their gradient (same layout)
  const float* mask;
};

template <typename T> struct TrainCtx {
  static constexpr bool k16 = !std::is_same<T, float>::value;
  Model& m;
  Arena& ar;
  cudaStream_t s;
  int H, I, heads, P;
  float eps;
  float p_hidden, p_attn;
  uint32_t step;
  uint64_t seed;
  float* G;
  uint32_t site = 0;  // dropout sites are numbered in forward order
  // backward scratch (take_backward)
  T *gT = nullptr, *gT2 = nullptr, *dmodBuf = nullptr, *trA = nullptr, *trB = nullptr;
  float* dmod32 = nullptr;
  const DropSpec nodrop{0.f, 0u, 0u, 0ull};

  TrainCtx(Model& m_, Arena& ar_, cudaStream_t s_, float ph, float pa, uint32_t st, uint64_t sd, float* g_)
      : m(m_), ar(ar_), s(s_), H(m_.cfg.hidden_size), I(m_.cfg.intermediate_size), heads(m_.cfg.num_attention_heads),
        P(m_.cfg.max_position_embeddings), eps(m_.cfg.layer_norm_eps), p_hidden(ph), p_attn(pa), step(st), seed(sd), G(g_) {}
  DropSpec hid() { return DropSpec{p_hidden, site++, step, seed}; }
  DropSpec att() { return DropSpec{p_attn, site++, step, seed}; }
  float* g(const std::string& n) const { return G + m.slots[m.slot_of.at(n)].off; }
  const Wt* rel(const AttnW& a) const { return m.cfg.relative_key ? &a.E : nullptr; }
  // gradient operands: gT / gT2 / dmodBuf / trA / trB elements, dmod32 floats
  void take_backward(size_t n_g, size_t n_mod, size_t n_trA, size_t n_trB, size_t n_mod32) {
    gT = ar.take<T>(n_g);        // gradient operand (dy of the Linear being differentiated)
    gT2 = ar.take<T>(n_g);       // second gradient operand (dx in T)
    dmodBuf = ar.take<T>(n_mod); // d(shift, scale, gate) of a per-token SELayer
    trA = ar.take<T>(n_trA);     // dy^T
    trB = ar.take<T>(n_trB);     // x^T
    dmod32 = ar.take<float>(n_mod32);
  }

  // ---- forward ------------------------------------------------------------------------------------
  // y (T) = x W^T + b
  int lin_T(int M, int N, int K, const T* X, const Wt& W, const float* bias, T* Y) {
    return gemm_any<T>(M, N, K, X, wsel<T>(W), bias, nullptr, Y, false, s);
  }
  // o (fp32) = dropout(x W^T + b) + resid
  int lin_res(int M, int N, int K, const T* X, const Wt& W, const float* bias, const float* resid, float* O, const DropSpec& dr) {
    if (dr.p <= 0.f) return gemm_any<T>(M, N, K, X, wsel<T>(W), bias, resid, O, true, s);
    SD_TRY(gemm_any<T>(M, N, K, X, wsel<T>(W), bias, nullptr, O, true, s));
    return dropout_add(O, resid, static_cast<size_t>(M) * N, dr, s);
  }
  // o = dropout(x W^T + b) + resid and h = LayerNorm(o): with dropout on, the residual add cannot ride in the GEMM epilogue (the mask sits
  // between the two), so it is folded into the LayerNorm pass instead of a pass of its own.
  int lin_res_ln(int M, int N, int K, const T* X, const Wt& W, const float* bias, const float* resid, float* O, const DropSpec& dr,
                 const float* ln_w, const float* ln_b, const Act2<T>& h, uint8_t* keep_bits) {
    if (dr.p > 0.f) {
      SD_TRY(gemm_any<T>(M, N, K, X, wsel<T>(W), bias, nullptr, O, true, s));
      return dropout_add_layernorm<T>(O, resid, dr, M, N, ln_w, ln_b, eps, h.s, h.t_out(), keep_bits, s);
    }
    SD_TRY(lin_res(M, N, K, X, W, bias, resid, O, dr));
    return layernorm<T>(O, M, N, ln_w, ln_b, eps, h.s, h.t_out(), nullptr, s);
  }
  // the attention dropout mask travels from the forward to the backward kernel as bits (2 KB per (graph, head)) when both run on the
  // tcgen05 kernels; every other combination regenerates it from the Philox stream
  uint32_t* keep_buf(int nb, int Lq, int Lk) {
    if (!k16 || p_attn <= 0.f || Lk % 4 != 0 || !attention_bwd_pipe_usable(Lq, Lk, nullptr, p_attn)) return nullptr;
    return ar.take<uint32_t>(static_cast<size_t>(nb) * heads * 128 * 4);
  }
  int attn_fwd(int nb, int Lq, int Lk, const T* q, int ldq, const T* k, int ldk, const T* v, int ldv, const Wt* E, const float* mask,
               const DropSpec& dr, T* out, uint32_t* keep) {
    const T* e = E ? static_cast<const T*>(wsel<T>(*E)) : nullptr;
    if (dr.p <= 0.f) return attention<T>(nb, heads, Lq, Lk, q, ldq, k, ldk, v, ldv, e, P, mask, out, s);
    if constexpr (k16) {
      // the pipelined tcgen05 kernel of the inference path with the dropout mask applied to P (7x faster than the wmma forward)
      if (Lk % 4 == 0) return attention_pipe_dropout<T>(nb, heads, Lq, Lk, q, ldq, k, ldk, v, ldv, e, P, mask, dr, out, s, keep);
      return attention_train_fwd_tc<T>(nb, heads, Lq, Lk, q, ldq, k, ldk, v, ldv, e, P, mask, dr, out, s);
    } else {
      return attention_train_fwd<T>(nb, heads, Lq, Lk, q, ldq, k, ldk, v, ldv, e, P, mask, dr, out, s);
    }
  }

  // SELayer (model.py:52-66) with its tape; tp.w, prefix, M, Mc, mod_div, x, c and segs are set by the caller
  int se_forward(SETape<T>& tp) {
    const SEW& w = *tp.w;
    const int M = tp.M, Mc = tp.Mc;
    const size_t MH = static_cast<size_t>(M) * H, McH = static_cast<size_t>(Mc) * H;
    tp.u_pre = ar.take<T>(McH);
    tp.u = ar.take<T>(McH);
    tp.mod = ar.take<T>(McH * 6);
    tp.qkv = ar.take<T>(MH * 3);
    tp.ctx = ar.take<T>(MH);
    tp.o = ar.take<float>(MH);
    tp.x1 = take_act2<T>(ar, MH);
    tp.m1_pre = ar.take<T>(MH * 4);
    tp.m1 = ar.take<T>(MH * 4);
    tp.m2 = ar.take<float>(MH);
    tp.out = take_act2<T>(ar, MH);
    tp.d_attn = att();
    tp.d_o = hid();
    tp.d_m1 = hid();
    tp.d_m2 = hid();
    SD_TRY(lin_T(Mc, H, H, tp.c, w.ada0, w.ada0_b, tp.u_pre));
    SD_TRY(act_fwd<T>(tp.u_pre, McH, 2, nodrop, tp.u, s));
    SD_TRY(lin_T(Mc, 6 * H, H, tp.u, w.ada2, w.ada2_b, tp.mod));
    SD_TRY(lin_T(M, 3 * H, H, tp.x.t, w.attn.qkv, w.attn.qkv_b, tp.qkv));
    for (const Segment& sg : tp.segs) {
      const T* base = tp.qkv + static_cast<size_t>(sg.row0) * 3 * H;
      DropSpec dr = tp.d_attn;
      tp.keep.push_back(keep_buf(sg.B, sg.L, sg.L));
      SD_TRY(attn_fwd(sg.B, sg.L, sg.L, base, 3 * H, base + H, 3 * H, base + 2 * H, 3 * H, rel(w.attn), sg.mask, dr,
                      tp.ctx + static_cast<size_t>(sg.row0) * H, tp.keep.back()));
    }
    SD_TRY(lin_res(M, H, H, tp.ctx, w.attn.out, w.attn.out_b, tp.x.s, tp.o, tp.d_o));
    SD_TRY(ln_modulate<T>(tp.o, M, H, true, w.attn.ln_w, w.attn.ln_b, eps, tp.x.s, tp.mod, tp.mod_div, 0, tp.x1.s, tp.x1.t_out(), s));
    SD_TRY(lin_T(M, 4 * H, H, tp.x1.t, w.m0, w.m0_b, tp.m1_pre));
    SD_TRY(act_fwd<T>(tp.m1_pre, MH * 4, 1, tp.d_m1, tp.m1, s));
    SD_TRY(lin_res(M, H, 4 * H, tp.m1, w.m3, w.m3_b, nullptr, tp.m2, tp.d_m2));
    SD_TRY(ln_modulate<T>(tp.m2, M, H, false, nullptr, nullptr, 0.f, tp.x1.s, tp.mod, tp.mod_div, 3, tp.out.s, tp.out.t_out(), s));
    return SEQDIFF_OK;
  }

  // HF BertLayer over B graphs of L rows (input h): self-attention (key mask `mask`) [-> cross-attention to *cr] -> FFN
  int layer_forward(LayerTape<T>& tp, const LayerW& w, int B, int L, const Act2<T>& h, const float* mask, const CrossKV<T>* cr) {
    const int M = B * L;
    const size_t MH = static_cast<size_t>(M) * H;
    tp.h = h;
    tp.qkv = ar.take<T>(MH * 3);
    tp.ctx = ar.take<T>(MH);
    tp.o1 = ar.take<float>(MH);
    tp.h1 = take_act2<T>(ar, MH);
    if (cr) {
      tp.cq = ar.take<T>(MH);
      tp.ctx2 = ar.take<T>(MH);
      tp.o2 = ar.take<float>(MH);
      tp.h2 = take_act2<T>(ar, MH);
    } else {
      tp.h2 = tp.h1;  // the FFN reads the self-attention sublayer's output
    }
    tp.f_pre = ar.take<T>(static_cast<size_t>(M) * I);
    tp.f = ar.take<T>(static_cast<size_t>(M) * I);
    tp.o3 = ar.take<float>(MH);
    tp.h3 = take_act2<T>(ar, MH);
    tp.d_attn = att();
    tp.d_o1 = hid();
    if (cr) {
      tp.d_cattn = att();
      tp.d_o2 = hid();
    }
    tp.d_o3 = hid();
    if (k16 && p_hidden > 0.f) {  // written by dropout_add_layernorm, read by the fused LayerNorm backward
      tp.kb1 = ar.take<uint8_t>(MH / 8);
      if (cr) tp.kb2 = ar.take<uint8_t>(MH / 8);
      tp.kb3 = ar.take<uint8_t>(MH / 8);
    }
    SD_TRY(lin_T(M, 3 * H, H, h.t, w.self.qkv, w.self.qkv_b, tp.qkv));
    tp.keep_self = keep_buf(B, L, L);
    SD_TRY(attn_fwd(B, L, L, tp.qkv, 3 * H, tp.qkv + H, 3 * H, tp.qkv + 2 * H, 3 * H, rel(w.self), mask, tp.d_attn, tp.ctx, tp.keep_self));
    SD_TRY(lin_res_ln(M, H, H, tp.ctx, w.self.out, w.self.out_b, h.s, tp.o1, tp.d_o1, w.self.ln_w, w.self.ln_b, tp.h1, tp.kb1));
    if (cr) {
      SD_TRY(lin_T(M, H, H, tp.h1.t, w.cq, w.cq_b, tp.cq));
      tp.keep_cross = keep_buf(B, L, cr->Lk);
      SD_TRY(attn_fwd(B, L, cr->Lk, tp.cq, H, cr->kv, cr->ld, cr->kv + H, cr->ld, nullptr, cr->mask, tp.d_cattn, tp.ctx2, tp.keep_cross));
      SD_TRY(lin_res_ln(M, H, H, tp.ctx2, w.cout, w.cout_b, tp.h1.s, tp.o2, tp.d_o2, w.cln_w, w.cln_b, tp.h2, tp.kb2));
    }
    SD_TRY(lin_T(M, I, H, tp.h2.t, w.inter, w.inter_b, tp.f_pre));
    SD_TRY(act_fwd<T>(tp.f_pre, static_cast<size_t>(M) * I, 1, nodrop, tp.f, s));
    SD_TRY(lin_res_ln(M, H, I, tp.f, w.outd, w.outd_b, tp.h2.s, tp.o3, tp.d_o3, w.oln_w, w.oln_b, tp.h3, tp.kb3));
    return SEQDIFF_OK;
  }

  // ---- backward -----------------------------------------------------------------------------------
  // backward of y = x W^T + b.  dY: T [M,N]; X: T [M,K].  dx_kind 0: none; 1: T [M,K]; 2: fp32 [M,K] (+ resid)
  // 16-bit modes: dW = dY^T X straight from the row-major tensors (both operands MN-major for the MMA, gemm_16_tn), db by a column-sum
  // kernel -- the two 16-bit transposes per Linear (11 % of the step) are gone.  fp32 mode and shapes failing tn_ok take the transposed form.
  bool tn_ok(int N, int K) const { return k16 && N % 8 == 0 && K % 128 == 0; }
  int linear_bwd(int M, int N, int K, const T* dY, const T* X, const Wt& W, float* gW, float* gb, int dx_kind, void* dX, const float* resid,
                 bool db_done = false) {
    if constexpr (k16) {
      if (tn_ok(N, K)) {
        if (!db_done) SD_TRY(colsum_add<T>(dY, M, N, gb, s));
        SD_TRY(gemm_16_tn(N, K, M, dY, X, TFmt<T>::v, m.d_zero_bias, gW, s, -1));  // split-K as below
        if (dx_kind) SD_TRY(gemm_any<T>(M, K, N, dY, W.t, m.d_zero_bias, resid, dX, dx_kind == 2, s));
        return SEQDIFF_OK;
      }
    }
    SD_CHECK(!db_done, "linear_bwd: fused bias gradient needs the in-place weight-gradient form");
    const int Mp = (M + 7) & ~7;  // contraction length of dW, padded with zero columns to a 16 B pitch
    SD_TRY(transpose_colsum<T>(dY, M, N, trA, gb, s, Mp));
    SD_TRY(transpose_colsum<T>(X, M, K, trB, nullptr, s, Mp));
    // dW [N,K]: a few dozen output tiles with a contraction over every token -> split-K over all SMs, partial products added
    // into the gradient buffer (zeroed at the start of the backward pass)
    SD_TRY(gemm_any<T>(N, K, Mp, trA, trB, m.d_zero_bias, nullptr, gW, true, s, -1));
    if (dx_kind) SD_TRY(gemm_any<T>(M, K, N, dY, W.t, m.d_zero_bias, resid, dX, dx_kind == 2, s));
    return SEQDIFF_OK;
  }
  int attn_bwd(int nb, int Lq, int Lk, const T* q, int ldq, const T* k, int ldk, const T* v, int ldv, const Wt* E, const float* mask,
               const DropSpec& dr, const T* dctx, T* dq, int lddq, T* dk, int lddk, T* dv, int lddv, float* gE, const uint32_t* keep) {
    const T* e = E ? static_cast<const T*>(wsel<T>(*E)) : nullptr;
    if constexpr (k16) {
      if (attention_bwd_pipe_usable(Lq, Lk, e, dr.p))  // tcgen05 backward
        return attention_bwd_pipe<T>(nb, heads, Lq, Lk, q, ldq, k, ldk, v, ldv, e, P, mask, dr, dctx, dq, lddq, dk, lddk, dv, lddv, gE, s, keep);
      return attention_bwd_tc<T>(nb, heads, Lq, Lk, q, ldq, k, ldk, v, ldv, e, P, mask, dr, dctx, dq, lddq, dk, lddk, dv, lddv, gE, s);
    } else {
      return attention_bwd<T>(nb, heads, Lq, Lk, q, ldq, k, ldk, v, ldv, e, P, mask, dr, dctx, dq, lddq, dk, lddk, dv, lddv, gE, s);
    }
  }

  // SELayer backward (model.py:52-63).  dout = gradient of tp.out.  Result: gradient of tp.x in s1; gradient of c in dc (if non-null).
  // tmp, s1, s2: fp32 [M,H] scratch, all distinct from dout.
  int se_backward(SETape<T>& tp, const float* dout, float* tmp, float* s1, float* s2, float* dc) {
    const SEW& w = *tp.w;
    const std::string p = tp.prefix;
    const int M = tp.M, Mc = tp.Mc;
    const size_t MH = static_cast<size_t>(M) * H, McH = static_cast<size_t>(Mc) * H;
    const bool per_tok = tp.mod_div == 1;
    T* dmT = per_tok ? dmodBuf : nullptr;
    float* dm32 = per_tok ? nullptr : dmod32;
    if (!per_tok) SD_CUDA(cudaMemsetAsync(dmod32, 0, McH * 6 * sizeof(float), s));
    // out = x1 + gate2 * (LN0(m2) * (1 + scale2) + shift2)
    SD_TRY(ln_modulate_bwd<T>(dout, tp.m2, M, H, false, nullptr, nullptr, 0.f, tp.mod, tp.mod_div, 3, s1, nullptr, dmT, dm32, nullptr, nullptr, s));
    SD_TRY(grad_cast<T>(s1, MH, tp.d_m2, gT, s));                                                     // d(m2) incl. its dropout mask
    SD_TRY(linear_bwd(M, H, 4 * H, gT, tp.m1, w.m3, g(p + ".mlp.3.weight"), g(p + ".mlp.3.bias"), 1, gT2, nullptr));  // d(m1)
    SD_TRY((act_bwd<T, T>(gT2, tp.m1_pre, MH * 4, 1, tp.d_m1, gT, s)));                                // d(m1_pre)
    SD_TRY(linear_bwd(M, 4 * H, H, gT, tp.x1.t, w.m0, g(p + ".mlp.0.weight"), g(p + ".mlp.0.bias"), 2, s1, dout));    // d(x1) = dout + ...
    // x1 = x + gate1 * (LN0(LN(o)) * (1 + scale1) + shift1);  o = dropout(ctx Wo^T + bo) + x
    SD_TRY(ln_modulate_bwd<T>(s1, tp.o, M, H, true, w.attn.ln_w, w.attn.ln_b, eps, tp.mod, tp.mod_div, 0, s2, tmp, dmT, dm32,
                              g(p + ".attn.output.LayerNorm.weight"), g(p + ".attn.output.LayerNorm.bias"), s));  // s2 = d(o); tmp = d(o) + d(x1)
    SD_TRY(grad_cast<T>(s2, MH, tp.d_o, gT, s));
    SD_TRY(linear_bwd(M, H, H, gT, tp.ctx, w.attn.out, g(p + ".attn.output.dense.weight"), g(p + ".attn.output.dense.bias"), 1, gT2, nullptr));  // d(ctx)
    for (size_t si = 0; si < tp.segs.size(); ++si) {
      const Segment& sg = tp.segs[si];
      const T* base = tp.qkv + static_cast<size_t>(sg.row0) * 3 * H;
      T* dbase = gT + static_cast<size_t>(sg.row0) * 3 * H;
      SD_TRY(attn_bwd(sg.B, sg.L, sg.L, base, 3 * H, base + H, 3 * H, base + 2 * H, 3 * H, rel(w.attn), sg.mask, tp.d_attn,
                      gT2 + static_cast<size_t>(sg.row0) * H, dbase, 3 * H, dbase + H, 3 * H, dbase + 2 * H, 3 * H,
                      m.cfg.relative_key ? g(p + ".attn.self.distance_embedding.weight") : nullptr, si < tp.keep.size() ? tp.keep[si] : nullptr));
    }
    SD_TRY(linear_bwd(M, 3 * H, H, gT, tp.x.t, w.attn.qkv, g(p + ".attn.self.query.weight"), g(p + ".attn.self.query.bias"), 2, s1, tmp));  // d(x)
    // adaLN_modulation: mod = Linear2(SiLU(Linear0(c)))
    const T* dmod = dmodBuf;
    if (!per_tok) {
      SD_TRY(grad_cast<T>(dmod32, McH * 6, nodrop, dmodBuf, s));
    }
    SD_TRY(linear_bwd(Mc, 6 * H, H, dmod, tp.u, w.ada2, g(p + ".adaLN_modulation.2.weight"), g(p + ".adaLN_modulation.2.bias"), 1, gT2, nullptr));  // d(u)
    SD_TRY((act_bwd<T, T>(gT2, tp.u_pre, McH, 2, nodrop, gT, s)));
    SD_TRY(linear_bwd(Mc, H, H, gT, tp.c, w.ada0, g(p + ".adaLN_modulation.0.weight"), g(p + ".adaLN_modulation.0.bias"), dc ? 2 : 0, dc, nullptr));
    return SEQDIFF_OK;
  }

  // post-LN sublayer h = LN(o), o = dropout(x W^T + b) + resid over M rows: d(o) in fp32 (it is also the gradient of resid) and, as the
  // Linear's dY, masked by the dropout site `dr` in the operand type (gT).  K = fan-in of that Linear (decides the weight-gradient form,
  // tn_ok).  (one launch: layernorm_bwd_cast also emits the 16-bit dY operand and the bias gradient of the Linear in front of it)
  bool ln_fused(int K) const { return tn_ok(H, K); }
  int ln_bwd(int M, const float* dh, const float* o, const float* gamma, float* d_o, float* dgam, float* dbet, const DropSpec& dr, float* dbias,
             int K, const uint8_t* keep_bits) {
    if constexpr (k16) {
      if (ln_fused(K)) return layernorm_bwd_cast<T>(dh, o, M, H, gamma, eps, d_o, dgam, dbet, dr, keep_bits, gT, dbias, s);
    }
    SD_TRY(layernorm_bwd(dh, o, M, H, gamma, eps, d_o, dgam, dbet, s));
    return grad_cast<T>(d_o, static_cast<size_t>(M) * H, dr, gT, s);
  }

  // backward of layer_forward.  dh = gradient of tp.h3 (read only); result: gradient of tp.h in s2.  s1, s2: fp32 [M,H] scratch.
  // The cross-attention's K | V gradient goes to cr->dkv.
  int layer_backward(LayerTape<T>& tp, const LayerW& w, const std::string& p, int B, int L, const float* mask, const CrossKV<T>* cr,
                     const float* dh, float* s1, float* s2) {
    const int M = B * L;
    const size_t MI = static_cast<size_t>(M) * I;
    // h3 = LN(o3); o3 = dropout(f Wod^T + b) + h2; f = GELU(h2 Wi^T + b)
    SD_TRY(ln_bwd(M, dh, tp.o3, w.oln_w, s1, g(p + ".output.LayerNorm.weight"), g(p + ".output.LayerNorm.bias"), tp.d_o3, g(p + ".output.dense.bias"), I,
                  tp.kb3));
    SD_TRY(linear_bwd(M, H, I, gT, tp.f, w.outd, g(p + ".output.dense.weight"), g(p + ".output.dense.bias"), 1, gT2, nullptr, ln_fused(I)));
    SD_TRY((act_bwd<T, T>(gT2, tp.f_pre, MI, 1, nodrop, gT, s)));
    SD_TRY(linear_bwd(M, I, H, gT, tp.h2.t, w.inter, g(p + ".intermediate.dense.weight"), g(p + ".intermediate.dense.bias"), 2, s2, s1));  // d(h2)
    if (cr) {
      // h2 = LN(o2); o2 = dropout(ctx2 Wco^T + b) + h1; ctx2 = cross-attention(q = h1 Wcq^T, k | v = receptor projections)
      SD_TRY(ln_bwd(M, s2, tp.o2, w.cln_w, s1, g(p + ".crossattention.output.LayerNorm.weight"), g(p + ".crossattention.output.LayerNorm.bias"),
                    tp.d_o2, g(p + ".crossattention.output.dense.bias"), H, tp.kb2));
      SD_TRY(linear_bwd(M, H, H, gT, tp.ctx2, w.cout, g(p + ".crossattention.output.dense.weight"), g(p + ".crossattention.output.dense.bias"), 1, gT2,
                        nullptr, ln_fused(H)));
      SD_TRY(attn_bwd(B, L, cr->Lk, tp.cq, H, cr->kv, cr->ld, cr->kv + H, cr->ld, nullptr, cr->mask, tp.d_cattn, gT2, gT, H, cr->dkv, cr->ld,
                      cr->dkv + H, cr->ld, nullptr, tp.keep_cross));
      SD_TRY(linear_bwd(M, H, H, gT, tp.h1.t, w.cq, g(p + ".crossattention.self.query.weight"), g(p + ".crossattention.self.query.bias"), 2, s2, s1));  // d(h1)
    }
    // h1 = LN(o1); o1 = dropout(ctx Wo^T + b) + h; ctx = self-attention(h Wqkv^T)
    SD_TRY(ln_bwd(M, s2, tp.o1, w.self.ln_w, s1, g(p + ".attention.output.LayerNorm.weight"), g(p + ".attention.output.LayerNorm.bias"), tp.d_o1,
                  g(p + ".attention.output.dense.bias"), H, tp.kb1));
    SD_TRY(linear_bwd(M, H, H, gT, tp.ctx, w.self.out, g(p + ".attention.output.dense.weight"), g(p + ".attention.output.dense.bias"), 1, gT2, nullptr,
                      ln_fused(H)));
    SD_TRY(attn_bwd(B, L, L, tp.qkv, 3 * H, tp.qkv + H, 3 * H, tp.qkv + 2 * H, 3 * H, rel(w.self), mask, tp.d_attn, gT2, gT, 3 * H, gT + H, 3 * H,
                    gT + 2 * H, 3 * H, m.cfg.relative_key ? g(p + ".attention.self.distance_embedding.weight") : nullptr, tp.keep_self));
    SD_TRY(linear_bwd(M, 3 * H, H, gT, tp.h.t, w.self.qkv, g(p + ".attention.self.query.weight"), g(p + ".attention.self.query.bias"), 2, s2, s1));  // d(h)
    return SEQDIFF_OK;
  }
};

static int ensure_train_workspace(Model& m, size_t need) {
  need = 2 * need + (64u << 20);  // the tape is carved out while kernels are already being launched: keep a wide safety margin
  if (need > m.tws_bytes) {
    if (m.tws) { SD_CUDA(cudaDeviceSynchronize()); debug_guard_begin(m.tws); SD_CUDA(cudaFree(m.tws)); m.tws = nullptr; m.tws_bytes = 0; }
    SD_CUDA(cudaMalloc(reinterpret_cast<void**>(&m.tws), need));
    m.tws_bytes = need;
  }
  return SEQDIFF_OK;
}

// =====================================================================================================
// one training step of the sequence model
// =====================================================================================================
template <typename T>
int Model::train_t(int wfmt, const TrainArgs& a, cudaStream_t s) {
  (void)wfmt;
  constexpr bool k16 = !std::is_same<T, float>::value;
  const int H = cfg.hidden_size, I = cfg.intermediate_size, NL = cfg.num_hidden_layers, heads = cfg.num_attention_heads;
  const int F = cfg.feature_size;
  const float eps = cfg.layer_norm_eps;
  const int B = a.B, Ll = a.Ll, Lr = a.Lr;
  const int Ml = B * Ll, Mr = B * Lr, Mt = Ml + Mr;
  const size_t MtH = static_cast<size_t>(Mt) * H, MlH = static_cast<size_t>(Ml) * H;
  SD_CHECK(Ml % 8 == 0 && Mr % 8 == 0, "training: B * L must be a multiple of 8 (vectorised rowwise kernels)");
  SD_CHECK(Ll <= 128 && Lr <= 128, "training: sequence length is limited to 128 (attention backward stages one key block)");
  const DropSpec nodrop{0.f, 0u, 0u, 0ull};

  // ---- workspace ----------------------------------------------------------------------------------
  const size_t es = sizeof(T);
  size_t need = 0;
  {
    const size_t act = al256(MtH * 4) + (k16 ? al256(MtH * 2) : 0);
    need += 8 * act;                                                  // x, c(32), x2, x1 (x2 SE layers), dec-norm out, spare
    need += 2 * (al256(MtH * es) * 3 + al256(MtH * 6 * es) + al256(MtH * 3 * es) + 2 * al256(MtH * 4 * es) + 2 * al256(MtH * 4));  // SE tapes
    need += al256(static_cast<size_t>(Mr) * NL * 2 * H * es) * 2;     // kv_all + its gradient
    need += static_cast<size_t>(NL) * (4 * act + al256(MlH * 3 * es) + 3 * al256(MlH * es) + 2 * al256(static_cast<size_t>(Ml) * I * es) + 3 * al256(MlH * 4));
    need += 3 * al256(MlH * es) + 2 * al256(static_cast<size_t>(Ml) * F * 4);  // head
    need += 6 * al256(MtH * 4);                                       // fp32 gradient streams
    need += 2 * al256(MtH * 6 * es) + al256(MtH * 6 * es) + al256(MtH * 4 * es);  // gradient operands + transposes
    need += al256(static_cast<size_t>(B) * 6 * H * 4) + 4 * al256(static_cast<size_t>(B) * 6 * H * es) + (1 << 20);
    need += static_cast<size_t>(2 * NL + 3) * al256(static_cast<size_t>(2 * B) * heads * 128 * 4 * sizeof(uint32_t));  // attention keep bits
    need += static_cast<size_t>(3 * NL) * al256(MlH / 8);             // hidden-dropout keep bits of the post-LN sublayers
  }
  SD_TRY(ensure_train_workspace(*this, need));
  Arena ar(tws, tws + tws_bytes, s);
  TrainCtx<T> cx(*this, ar, s, a.p_hidden, a.p_attn, a.step, a.seed, a.grads);
  auto g = [&](const std::string& n) { return cx.g(n); };

  // ---- forward ------------------------------------------------------------------------------------
  float* te = ar.take<float>(static_cast<size_t>(B) * H);
  T* teT = k16 ? ar.take<T>(static_cast<size_t>(B) * H) : reinterpret_cast<T*>(te);
  float* maskcat = ar.take<float>(static_cast<size_t>(Mt));
  SD_TRY(timestep_embed(a.t_norm, nullptr, ts_W, B, H, te, k16 ? static_cast<void*>(teT) : nullptr, TFmt<T>::v, s));
  Act2<T> x = take_act2<T>(ar, MtH);
  float* c32 = ar.take<float>(MtH);
  T* ccat = k16 ? ar.take<T>(MtH) : reinterpret_cast<T*>(c32);
  const DropSpec d_emb[4] = {cx.hid(), cx.hid(), cx.hid(), cx.hid()};  // lig seq, rec seq, lig angle, rec angle
  {
    auto job = [&](const float* in, int M, const EmbW& e, const float* te_, int L, float* o32, T* oT) {
      EmbedJob jb{};
      jb.x = in; jb.Wt = e.Wt_; jb.b = e.b; jb.lnw = e.ln_w; jb.lnb = e.ln_b; jb.te = te_;
      jb.out32 = o32; jb.outT = oT; jb.M = M; jb.fin = e.fin; jb.L = L;
      return jb;
    };
    const bool dropping = a.p_hidden > 0.f;
    EmbedJobs jobs{};
    jobs.n = 4;
    jobs.j[0] = job(a.x_t, Ml, lig_seq, nullptr, Ll, x.s, dropping ? nullptr : x.t_out());
    jobs.j[1] = job(a.rec_seq, Mr, rec_seq, nullptr, Lr, x.s + MlH, dropping ? nullptr : (k16 ? x.t + MlH : nullptr));
    jobs.j[2] = job(a.lig_angle, Ml, lig_ang, dropping ? nullptr : te, Ll, c32, (dropping || !k16) ? nullptr : ccat);
    jobs.j[3] = job(a.rec_angle, Mr, rec_ang, dropping ? nullptr : te, Lr, c32 + MlH, (dropping || !k16) ? nullptr : ccat + MlH);
    SD_TRY(embed_ln_multi<T>(jobs, eps, H, s));
    if (dropping) {
      SD_TRY(embed_post<T>(x.s, nullptr, Ll, H, MlH, d_emb[0], x.s, x.t, s));
      SD_TRY(embed_post<T>(x.s + MlH, nullptr, Lr, H, static_cast<size_t>(Mr) * H, d_emb[1], x.s + MlH, x.t + MlH, s));
      SD_TRY(embed_post<T>(c32, te, Ll, H, MlH, d_emb[2], c32, ccat, s));
      SD_TRY(embed_post<T>(c32 + MlH, te, Lr, H, static_cast<size_t>(Mr) * H, d_emb[3], c32 + MlH, ccat + MlH, s));
    }
    SD_CUDA(launch_k(concat_masks_kernel, dim3(32), dim3(256), 0, s, maskcat, a.lig_mask, Ml, a.rec_mask, Mr));
    SD_LAUNCHED("concat_masks", s);
  }

  // ligand_feature_emb over [ligand | receptor] tokens (quirk Q1)
  SETape<T> se1;
  se1.w = &se_lig;
  se1.prefix = "ligand_feature_emb";
  se1.M = Mt; se1.Mc = Mt; se1.mod_div = 1;
  se1.x = x;
  se1.c = ccat;
  if (Ll == Lr) {
    se1.segs.push_back({0, 2 * B, Ll, maskcat});
  } else {
    se1.segs.push_back({0, B, Ll, a.lig_mask});
    se1.segs.push_back({Ml, B, Lr, a.rec_mask});
  }
  SD_TRY(cx.se_forward(se1));
  const T* rec_t = se1.out.t + MlH;

  // decoder
  T* kv_all = ar.take<T>(static_cast<size_t>(Mr) * NL * 2 * H);
  SD_TRY(cx.lin_T(Mr, NL * 2 * H, H, rec_t, ckv_all, ckv_all_b, kv_all));
  std::vector<LayerTape<T>> lt(NL);
  std::vector<CrossKV<T>> ckv(NL);
  Act2<T> h = se1.out;  // ligand rows = first Ml rows
  for (int i = 0; i < NL; ++i) {
    ckv[i] = CrossKV<T>{Lr, NL * 2 * H, kv_all + static_cast<size_t>(i) * 2 * H, nullptr, a.rec_mask};
    SD_TRY(cx.layer_forward(lt[i], layers[i], B, Ll, h, a.lig_mask, &ckv[i]));
    h = lt[i].h3;
  }

  // decoder_normalize (c = timestep features, broadcast over the graph)
  SETape<T> se2;
  se2.w = &se_dec;
  se2.prefix = "decoder_normalize";
  se2.M = Ml; se2.Mc = B; se2.mod_div = Ll;
  se2.x = h;
  se2.c = teT;
  se2.segs.push_back({0, B, Ll, a.lig_mask});
  SD_TRY(cx.se_forward(se2));

  // head + loss
  T* z1 = ar.take<T>(MlH);
  T* y = ar.take<T>(MlH);
  float* logits = a.logits_out ? a.logits_out : ar.take<float>(static_cast<size_t>(Ml) * F);
  float* dlogits = ar.take<float>(static_cast<size_t>(Ml) * F);
  SD_TRY(cx.lin_T(Ml, H, H, se2.out.t, p1, p1_b, z1));
  SD_TRY(act_fwd<T>(z1, MlH, 1, nodrop, y, s));
  SD_TRY(predictor_tail<T>(y, Ml, H, p_ln_w, p_ln_b, 1e-12f, p2_w, p2_b, F, logits, s));
  double* loss_scratch = ar.take<double>(loss_terms_scratch_bytes() / sizeof(double));  // no allocator call inside the step
  SD_CHECK(ar.ok, "training workspace under-estimated");
  SD_TRY(loss_terms(Ml, logits, a.x0, a.x_t, a.lig_mask, a.terms, s, loss_scratch));
  SD_TRY(loss_bwd(Ml, logits, a.x0, a.x_t, a.terms, dlogits, s));

  // ---- backward -----------------------------------------------------------------------------------
  SD_CUDA(cudaMemsetAsync(a.grads, 0, static_cast<size_t>(train_total) * sizeof(float), s));
  float* dA = ar.take<float>(MtH);
  float* dB = ar.take<float>(MtH);
  float* dC = ar.take<float>(MtH);
  float* dD = ar.take<float>(MtH);
  float* dc32 = ar.take<float>(MtH);
  T* dkv_all = ar.take<T>(static_cast<size_t>(Mr) * NL * 2 * H);
  cx.take_backward(MtH * 6, MtH * 6, MtH * 6, MtH * 4, static_cast<size_t>(B) * 6 * H);
  SD_CHECK(ar.ok, "training workspace under-estimated");
  T* gT = cx.gT;

  // head: logits = LN(GELU(x W1^T + b1)) W2^T + b2
  const std::string hp = "amino_acid_predictor.";
  SD_TRY(predictor_tail_bwd<T>(dlogits, y, Ml, H, p_ln_w, p_ln_b, 1e-12f, p2_w, F, dA, g(hp + "dense2.weight"), g(hp + "dense2.bias"),
                               g(hp + "layer_norm.weight"), g(hp + "layer_norm.bias"), s));
  if constexpr (k16) {
    SD_TRY((act_bwd<T, float>(dA, z1, MlH, 1, nodrop, gT, s)));
  } else {
    SD_TRY((act_bwd<float, float>(dA, z1, MlH, 1, nodrop, gT, s)));
  }
  SD_TRY(cx.linear_bwd(Ml, H, H, gT, se2.out.t, p1, g(hp + "dense1.weight"), g(hp + "dense1.bias"), 2, dB, nullptr));
  // decoder_normalize
  SD_TRY(cx.se_backward(se2, dB, dC, dA, dD, nullptr));  // d(h_last) in dA
  const int n_bk = static_cast<int>(grad_bucket_bounds.size()) - 1;
  auto bucket_done = [&](int k) -> int {  // gradients of flat range [bounds[k], bounds[k+1]) are final from here on
    if (k >= 0 && k < static_cast<int>(bucket_events.size()) && bucket_events[k]) SD_CUDA(cudaEventRecord(bucket_events[k], s));
    return SEQDIFF_OK;
  };
  SD_TRY(bucket_done(n_bk - 1));
  // decoder layers, last to first
  float *cur = dA, *s1 = dB, *s2 = dC;
  for (int i = NL - 1; i >= 0; --i) {
    ckv[i].dkv = dkv_all + static_cast<size_t>(i) * 2 * H;
    SD_TRY(cx.layer_backward(lt[i], layers[i], "decoder.layer." + std::to_string(i), B, Ll, a.lig_mask, &ckv[i], cur, s1, s2));
    float* t_ = cur;
    cur = s2;
    s2 = t_;
    if (n_bk == 4 && i == NL / 2) SD_TRY(bucket_done(2));
  }
  // gradient of ligand_feature_emb's output: [d(ligand rows) ; d(receptor rows)], the latter through the fused cross K | V projection
  SD_CUDA(cudaMemcpyAsync(dD, cur, MlH * sizeof(float), cudaMemcpyDeviceToDevice, s));
  SD_TRY(cx.linear_bwd(Mr, NL * 2 * H, H, dkv_all, rec_t, ckv_all, g("decoder.layer.0.crossattention.self.key.weight"),
                       g("decoder.layer.0.crossattention.self.key.bias"), 2, dD + MlH, nullptr));
  SD_TRY(bucket_done(1));
  SD_TRY(cx.se_backward(se1, dD, dC, dA, dB, dc32));  // d(x) in dA, d(c) in dc32
  // the four BertEmbeddings
  SD_TRY(embed_bwd(dA, a.x_t, Ml, 20, H, lig_seq.Wt_, lig_seq.b, lig_seq.ln_w, eps, d_emb[0], g("ligand_seq_embedding.linear.weight"),
                   g("ligand_seq_embedding.linear.bias"), g("ligand_seq_embedding.LayerNorm.weight"), g("ligand_seq_embedding.LayerNorm.bias"), s));
  SD_TRY(embed_bwd(dA + MlH, a.rec_seq, Mr, 20, H, rec_seq.Wt_, rec_seq.b, rec_seq.ln_w, eps, d_emb[1], g("receptor_seq_embedding.linear.weight"),
                   g("receptor_seq_embedding.linear.bias"), g("receptor_seq_embedding.LayerNorm.weight"), g("receptor_seq_embedding.LayerNorm.bias"), s));
  SD_TRY(embed_bwd(dc32, a.lig_angle, Ml, 8, H, lig_ang.Wt_, lig_ang.b, lig_ang.ln_w, eps, d_emb[2], g("ligand_angle_embedding.linear.weight"),
                   g("ligand_angle_embedding.linear.bias"), g("ligand_angle_embedding.LayerNorm.weight"), g("ligand_angle_embedding.LayerNorm.bias"), s));
  SD_TRY(embed_bwd(dc32 + MlH, a.rec_angle, Mr, 8, H, rec_ang.Wt_, rec_ang.b, rec_ang.ln_w, eps, d_emb[3], g("receptor_angle_embedding.linear.weight"),
                   g("receptor_angle_embedding.linear.bias"), g("receptor_angle_embedding.LayerNorm.weight"), g("receptor_angle_embedding.LayerNorm.bias"), s));
  SD_TRY(bucket_done(0));
  return SEQDIFF_OK;
}

// =====================================================================================================
// one training step of the structure (angle) model: structure_model/model.py:180-215 in training mode + the wrapped smooth-L1
// objective on the predicted noise (decode_loss.cu: angle_loss_terms) + the full backward
// =====================================================================================================
template <typename T>
int Model::struct_train_t(const StructTrainArgs& a, cudaStream_t s) {
  constexpr bool k16 = !std::is_same<T, float>::value;
  const int H = cfg.hidden_size, I = cfg.intermediate_size, NL = cfg.num_hidden_layers, heads = cfg.num_attention_heads;
  const int F = cfg.feature_size;
  const float eps = cfg.layer_norm_eps;
  const int B = a.B, Ll = a.Ll, Lr = a.Lr;
  const int Ml = B * Ll, Mr = B * Lr, Mx = Ml > Mr ? Ml : Mr;
  const size_t MlH = static_cast<size_t>(Ml) * H, MrH = static_cast<size_t>(Mr) * H, MxH = static_cast<size_t>(Mx) * H;
  const DropSpec nodrop{0.f, 0u, 0u, 0ull};

  // ---- workspace ----------------------------------------------------------------------------------
  const size_t es = sizeof(T);
  const size_t n_op = MxH * 6 > static_cast<size_t>(Mx) * I ? MxH * 6 : static_cast<size_t>(Mx) * I;  // widest [M, N] gradient operand
  const size_t n_kv = static_cast<size_t>(Mr) * NL * 2 * H;
  const size_t n_trA = n_op > n_kv ? n_op : n_kv;
  size_t need = 0;
  {
    const size_t act = al256(MxH * 4) + (k16 ? al256(MxH * 2) : 0);
    need += 6 * act + 2 * al256(static_cast<size_t>(B) * H * 4);     // embeddings, c, timestep features
    need += 2 * (al256(MxH * es) * 3 + al256(MxH * 6 * es) + al256(MxH * 3 * es) + 2 * al256(MxH * 4 * es) + 2 * al256(MxH * 4) + 2 * act);  // SE tapes
    need += 2 * al256(n_kv * es);                                     // kv_all + its gradient
    const size_t per_layer = 4 * act + al256(MxH * 3 * es) + 3 * al256(MxH * es) + 2 * al256(static_cast<size_t>(Mx) * I * es) + 3 * al256(MxH * 4) +
                             3 * al256(MxH / 8) + 2 * al256(static_cast<size_t>(2 * B) * heads * 128 * 4 * sizeof(uint32_t));
    need += static_cast<size_t>(2 * NL) * per_layer;                  // encoder + decoder tapes
    need += 2 * al256(MlH * es) + 3 * al256(static_cast<size_t>(Ml) * F * 4) + al256(angle_loss_scratch_bytes());  // head + loss
    need += 6 * al256(MxH * 4);                                       // fp32 gradient streams
    need += 2 * al256(n_op * es) + al256(MxH * 6 * es) + al256(n_trA * es) + al256(n_op * es);  // gradient operands + transposes
    need += al256(static_cast<size_t>(B) * 6 * H * 4) + (1 << 20);
  }
  SD_TRY(ensure_train_workspace(*this, need));
  Arena ar(tws, tws + tws_bytes, s);
  TrainCtx<T> cx(*this, ar, s, a.p_hidden, a.p_attn, a.step, a.seed, a.grads);
  auto g = [&](const std::string& n) { return cx.g(n); };

  // ---- forward ------------------------------------------------------------------------------------
  // embeddings (BertEmbeddings: LN(Linear(x)), then its dropout): receptor angles -> x, receptor sequence -> c, ligand angles -> x
  float* te = ar.take<float>(static_cast<size_t>(B) * H);
  T* teT = k16 ? ar.take<T>(static_cast<size_t>(B) * H) : reinterpret_cast<T*>(te);
  SD_TRY(timestep_embed(a.t, nullptr, ts_W, B, H, te, k16 ? static_cast<void*>(teT) : nullptr, TFmt<T>::v, s));
  Act2<T> xr = take_act2<T>(ar, MrH);
  Act2<T> cr = take_act2<T>(ar, MrH);
  Act2<T> xl = take_act2<T>(ar, MlH);
  const DropSpec d_emb[3] = {cx.hid(), cx.hid(), cx.hid()};  // receptor angle, receptor seq, ligand angle
  {
    auto job = [&](const float* in, int M, const EmbW& e, int L, const Act2<T>& o) {
      EmbedJob jb{};
      jb.x = in; jb.Wt = e.Wt_; jb.b = e.b; jb.lnw = e.ln_w; jb.lnb = e.ln_b; jb.te = nullptr;
      jb.out32 = o.s; jb.outT = a.p_hidden > 0.f ? nullptr : o.t_out(); jb.M = M; jb.fin = e.fin; jb.L = L;
      return jb;
    };
    EmbedJobs jobs{};
    jobs.n = 3;
    jobs.j[0] = job(a.rec_angle, Mr, rec_ang, Lr, xr);
    jobs.j[1] = job(a.rec_seq, Mr, rec_seq, Lr, cr);
    jobs.j[2] = job(a.corrupted, Ml, lig_ang, Ll, xl);
    SD_TRY(embed_ln_multi<T>(jobs, eps, H, s));
    if (a.p_hidden > 0.f) {
      SD_TRY(embed_post<T>(xr.s, nullptr, Lr, H, MrH, d_emb[0], xr.s, xr.t, s));
      SD_TRY(embed_post<T>(cr.s, nullptr, Lr, H, MrH, d_emb[1], cr.s, cr.t, s));
      SD_TRY(embed_post<T>(xl.s, nullptr, Ll, H, MlH, d_emb[2], xl.s, xl.t, s));
    }
  }
  // receptor branch: receptor_emb (x = angles, c = sequence, per token), the encoder, every decoder layer's cross K | V in one GEMM
  SETape<T> se1;
  se1.w = &se_lig;
  se1.prefix = "receptor_emb";
  se1.M = Mr; se1.Mc = Mr; se1.mod_div = 1;
  se1.x = xr;
  se1.c = cr.t;
  se1.segs.push_back({0, B, Lr, a.rec_mask});
  SD_TRY(cx.se_forward(se1));
  std::vector<LayerTape<T>> et(NL);
  Act2<T> h = se1.out;
  for (int i = 0; i < NL; ++i) {
    SD_TRY(cx.layer_forward(et[i], enc_layers[i], B, Lr, h, a.rec_mask, nullptr));
    h = et[i].h3;
  }
  const Act2<T> enc_out = h;
  T* kv_all = ar.take<T>(n_kv);
  SD_TRY(cx.lin_T(Mr, NL * 2 * H, H, enc_out.t, ckv_all, ckv_all_b, kv_all));
  // ligand branch: timestep_emb (c = timestep features, broadcast over the graph), the decoder, the head
  SETape<T> se2;
  se2.w = &se_dec;
  se2.prefix = "timestep_emb";
  se2.M = Ml; se2.Mc = B; se2.mod_div = Ll;
  se2.x = xl;
  se2.c = teT;
  se2.segs.push_back({0, B, Ll, a.lig_mask});
  SD_TRY(cx.se_forward(se2));
  std::vector<LayerTape<T>> lt(NL);
  std::vector<CrossKV<T>> ckv(NL);
  h = se2.out;
  for (int i = 0; i < NL; ++i) {
    ckv[i] = CrossKV<T>{Lr, NL * 2 * H, kv_all + static_cast<size_t>(i) * 2 * H, nullptr, a.rec_mask};
    SD_TRY(cx.layer_forward(lt[i], layers[i], B, Ll, h, a.lig_mask, &ckv[i]));
    h = lt[i].h3;
  }
  T* z1 = ar.take<T>(MlH);
  T* y = ar.take<T>(MlH);
  float* pred = a.pred_out ? a.pred_out : ar.take<float>(static_cast<size_t>(Ml) * F);
  float* dpred = ar.take<float>(static_cast<size_t>(Ml) * F);
  SD_TRY(cx.lin_T(Ml, H, H, h.t, p1, p1_b, z1));
  SD_TRY(act_fwd<T>(z1, MlH, 1, nodrop, y, s));
  SD_TRY(predictor_tail<T>(y, Ml, H, p_ln_w, p_ln_b, 1e-12f, p2_w, p2_b, F, pred, s));
  double* loss_scratch = ar.take<double>(angle_loss_scratch_bytes() / sizeof(double));  // no allocator call inside the step
  SD_CHECK(ar.ok, "training workspace under-estimated");
  SD_TRY(angle_loss_terms(Ml, F, pred, a.known_noise, a.lig_mask, a.terms, s, loss_scratch));
  SD_TRY(angle_loss_bwd(Ml, F, pred, a.known_noise, a.lig_mask, a.terms, dpred, s));

  // ---- backward -----------------------------------------------------------------------------------
  SD_CUDA(cudaMemsetAsync(a.grads, 0, static_cast<size_t>(train_total) * sizeof(float), s));
  float* dA = ar.take<float>(MxH);
  float* dB = ar.take<float>(MxH);
  float* dC = ar.take<float>(MxH);
  float* dD = ar.take<float>(MxH);
  float* dc32 = ar.take<float>(MrH);
  cx.take_backward(n_op, MxH * 6, n_trA, n_op, static_cast<size_t>(B) * 6 * H);
  T* dkv_all = ar.take<T>(n_kv);
  SD_CHECK(ar.ok, "training workspace under-estimated");
  T* gT = cx.gT;
  const int n_bk = static_cast<int>(grad_bucket_bounds.size()) - 1;
  int bk = n_bk - 1;
  auto bucket_done = [&]() -> int {  // the next bucket from the end is final from here on (bounds: build_slots)
    const int k = bk--;
    if (k >= 0 && k < static_cast<int>(bucket_events.size()) && bucket_events[k]) SD_CUDA(cudaEventRecord(bucket_events[k], s));
    return SEQDIFF_OK;
  };
  const bool halves = NL >= 2;  // build_slots splits both stacks in halves then
  // head: pred = LN(GELU(h W1^T + b1)) W2^T + b2
  const std::string hp = "angles_predictor.";
  SD_TRY(predictor_tail_bwd<T>(dpred, y, Ml, H, p_ln_w, p_ln_b, 1e-12f, p2_w, F, dA, g(hp + "dense2.weight"), g(hp + "dense2.bias"),
                               g(hp + "layer_norm.weight"), g(hp + "layer_norm.bias"), s));
  if constexpr (k16) {
    SD_TRY((act_bwd<T, float>(dA, z1, MlH, 1, nodrop, gT, s)));
  } else {
    SD_TRY((act_bwd<float, float>(dA, z1, MlH, 1, nodrop, gT, s)));
  }
  SD_TRY(cx.linear_bwd(Ml, H, H, gT, h.t, p1, g(hp + "dense1.weight"), g(hp + "dense1.bias"), 2, dB, nullptr));
  // decoder layers, last to first
  float *cur = dB, *s1 = dA, *s2 = dC;
  for (int i = NL - 1; i >= 0; --i) {
    ckv[i].dkv = dkv_all + static_cast<size_t>(i) * 2 * H;
    SD_TRY(cx.layer_backward(lt[i], layers[i], "decoder.layer." + std::to_string(i), B, Ll, a.lig_mask, &ckv[i], cur, s1, s2));
    std::swap(cur, s2);
    if (halves && i == NL / 2) SD_TRY(bucket_done());
  }
  // timestep_emb: the timestep features take no gradient (timestep_projector.W is a buffer); then ligand_angle_emb
  SD_TRY(cx.se_backward(se2, cur, s2, s1, dD, nullptr));  // d(x) in s1
  SD_TRY(embed_bwd(s1, a.corrupted, Ml, F, H, lig_ang.Wt_, lig_ang.b, lig_ang.ln_w, eps, d_emb[2], g("ligand_angle_emb.linear.weight"),
                   g("ligand_angle_emb.linear.bias"), g("ligand_angle_emb.LayerNorm.weight"), g("ligand_angle_emb.LayerNorm.bias"), s));
  // gradient of the encoder output: every decoder layer's K | V gradient through the fused projection, in one GEMM
  cur = dA;
  s1 = dB;
  s2 = dC;
  SD_TRY(cx.linear_bwd(Mr, NL * 2 * H, H, dkv_all, enc_out.t, ckv_all, g("decoder.layer.0.crossattention.self.key.weight"),
                       g("decoder.layer.0.crossattention.self.key.bias"), 2, cur, nullptr));
  SD_TRY(bucket_done());
  // encoder layers, last to first
  for (int i = NL - 1; i >= 0; --i) {
    SD_TRY(cx.layer_backward(et[i], enc_layers[i], "encoder.layer." + std::to_string(i), B, Lr, a.rec_mask, nullptr, cur, s1, s2));
    std::swap(cur, s2);
    if (halves && i == NL / 2) SD_TRY(bucket_done());
  }
  // receptor_emb (per-token c = the receptor sequence embedding), then the two receptor embeddings
  SD_TRY(cx.se_backward(se1, cur, s2, s1, dD, dc32));  // d(x) in s1, d(c) in dc32
  SD_TRY(embed_bwd(dc32, a.rec_seq, Mr, 20, H, rec_seq.Wt_, rec_seq.b, rec_seq.ln_w, eps, d_emb[1], g("receptor_seq_emb.linear.weight"),
                   g("receptor_seq_emb.linear.bias"), g("receptor_seq_emb.LayerNorm.weight"), g("receptor_seq_emb.LayerNorm.bias"), s));
  SD_TRY(embed_bwd(s1, a.rec_angle, Mr, F, H, rec_ang.Wt_, rec_ang.b, rec_ang.ln_w, eps, d_emb[0], g("receptor_angle_emb.linear.weight"),
                   g("receptor_angle_emb.linear.bias"), g("receptor_angle_emb.LayerNorm.weight"), g("receptor_angle_emb.LayerNorm.bias"), s));
  SD_TRY(bucket_done());
  return SEQDIFF_OK;
}

// Programmatic dependent launch of the heavy kernels of a training step (mode 3: tcgen05 GEMMs and attention -- their prologue, i.e.
// barrier init, TMEM allocation, descriptor prefetch, runs under the predecessor's tail).  Every kernel launched inside the step starts
// with griddepcontrol.wait, so any mode is safe.  Measured on B200 (profiles/train_pdl_ab_r02.log): 128 graphs 15.15 -> 14.64 ms per
// step, 16 graphs 5.00 -> 4.55 ms; every launch (mode 1) 14.72 / 4.76 ms.
struct TrainPdlScope {
  const int prev;
  explicit TrainPdlScope(int m) : prev(pdl_scope_exchange(m)) {}
  ~TrainPdlScope() { pdl_scope_exchange(prev); }
};

// checks shared by both steps; builds the parameter table and, on the first call or a precision switch, the transposed operand copies
int Model::train_prologue(int precision, int B, int Ll, int Lr, float p_hidden, float p_attn, cudaStream_t s) {
  SD_CHECK(finalized, "model not finalised (seqdiff_model_finalize)");
  SD_CHECK(precision >= SEQDIFF_FP32 && precision <= SEQDIFF_FP16, "unknown precision mode");
  SD_CHECK(B > 0 && Ll > 0 && Lr > 0, "empty batch");
  SD_CHECK(p_hidden >= 0.f && p_hidden < 1.f && p_attn >= 0.f && p_attn < 1.f, "dropout probabilities must be in [0, 1)");
  if (cfg.relative_key) SD_CHECK(Ll <= cfg.max_position_embeddings && Lr <= cfg.max_position_embeddings, "Length exceed");
  SD_CUDA(cudaSetDevice(device));
  SD_TRY(build_slots());
  if (train_prec != precision) {  // first training call (or a precision switch): build the transposed operand copies
    train_prec = precision;
    SD_TRY(finalize(s));
  }
  if (g_profiling) profile_mark("__begin__", s);  // host time between two steps is not the first kernel's
  return SEQDIFF_OK;
}

int Model::train_step(const TrainArgs& a, cudaStream_t s) {
  SD_CHECK(arch == kArchSequence, "handle holds a structure model: use seqdiff_struct_train_step");
  SD_CHECK(cfg.feature_size == SEQDIFF_NUM_CLASSES, "training needs feature_size == 20");
  SD_TRY(train_prologue(a.precision, a.B, a.Ll, a.Lr, a.p_hidden, a.p_attn, s));
  TrainPdlScope pdl_scope(3);
  switch (a.precision) {
    case SEQDIFF_FP32: return train_t<float>(1, a, s);
    case SEQDIFF_BF16: return train_t<bf16>(1, a, s);
    default: return train_t<f16>(0, a, s);
  }
}

int Model::struct_train_step(const StructTrainArgs& a, cudaStream_t s) {
  SD_CHECK(arch == kArchStructure, "handle holds a sequence model: use seqdiff_train_step");
  SD_CHECK(cfg.feature_size == 8 || cfg.feature_size == 20, "structure training needs feature_size 8 or 20 (angle head backward)");
  SD_CHECK(a.B * a.Ll % 8 == 0 && a.B * a.Lr % 8 == 0, "training: B * L must be a multiple of 8 (vectorised rowwise kernels)");
  SD_CHECK(a.Ll <= 128 && a.Lr <= 128, "training: sequence length is limited to 128 (attention backward stages one key block)");
  SD_TRY(train_prologue(a.precision, a.B, a.Ll, a.Lr, a.p_hidden, a.p_attn, s));
  TrainPdlScope pdl_scope(3);
  switch (a.precision) {
    case SEQDIFF_FP32: return struct_train_t<float>(a, s);
    case SEQDIFF_BF16: return struct_train_t<bf16>(a, s);
    default: return struct_train_t<f16>(a, s);
  }
}

}  // namespace seqdiff
