// kernels.h -- internal launcher interface between the kernel translation units and model.cu/cabi.cu.
// Every function enqueues on `s`, returns SEQDIFF_OK or an error code (message via set_error()).
#pragma once
#include "common.cuh"
#include "philox.cuh"

namespace seqdiff {

// ---- gemm.cu ----------------------------------------------------------------------------------------
// epi: 0 identity, 1 erf-GELU, 2 SiLU.  resid (same shape as C) only with epi == 0.
// tcgen05 GEMM on 16-bit operands.  a_fmt / w_fmt: 0 = fp16, 1 = bf16.  out_kind: 0 = fp16, 1 = bf16, 2 = fp32.
// resid is fp32 and implies an fp32 output (the residual stream never takes a 16-bit rounding).
// ln_resid != NULL: the residual is LayerNorm(resid) = (resid - mean) * rstd * g + b rebuilt on the fly (see LnResid).
struct LnResid {
  const float2* stats;  // [M] (mean, rstd) written by layernorm()
  const float* g;       // [N] LayerNorm weight
  const float* b;       // [N] LayerNorm bias
};
// ln_out != NULL (needs resid, fp32 C, N in {512, 768, 1024}): the kernel also applies the LayerNorm that FOLLOWS this
// Linear -- h = LN(C) * g + b written as the 16-bit operand of the next GEMM, (mean, rstd) per row for a later LnResid
// rebuild -- so the separate layernorm() launch and its re-read of C disappear.  Four CTAs of a cluster cover the 4 column
// quarters of a 128-row block and exchange per-row partial sums through distributed shared memory.
struct LnOut {
  const float* g;   // [N] LayerNorm weight
  const float* b;   // [N] LayerNorm bias
  float eps;
  void* h;          // [M, N] 16-bit output (format = a_fmt)
  float2* stats;    // [M] (mean, rstd)
};
int gemm_16(int M, int N, int K, const void* A, int a_fmt, const void* W, int w_fmt, const float* bias, const float* resid, int epi,
            void* C, int out_kind, cudaStream_t s, int force_bn = 0, const LnResid* ln_resid = nullptr, const LnOut* ln_out = nullptr,
            int split_k = 1);  // split_k: 1 off | n k-ranges per tile | -1 auto; partial products are ADDED into a pre-zeroed fp32 C
// C[M,N] (+)= At^T Bt + bias: At [K, M], Bt [K, N] row-major 16-bit (both MN-major for the MMA: no transposed copies); fp32 C.
// The weight-gradient product dW[N_out, N_in] = dY^T X of the training step (At = dY [tokens, N_out], Bt = X [tokens, N_in]).
int gemm_16_tn(int M, int N, int K, const void* At, const void* Bt, int fmt, const float* bias, float* C, cudaStream_t s, int split_k = 1);
int gemm_f32(int M, int N, int K, const float* A, const float* W, const float* bias, const float* resid, int epi, float* C,
             cudaStream_t s);

// TMA descriptor (cached) of a row-major 16-bit matrix [rows, cols]: boxes of box_rows x 64 columns, 128B swizzle, OOB -> 0
int make_tmap(const void* ptr, int fmt, int rows, int cols, int box_rows, CUtensorMap* out);
// [batch][rows][cols] variant (uncached) for per-graph TMA stores: boxes of 1 x box_rows x 64, rows clipped per graph
int make_tmap_3d(const void* ptr, int fmt, int batch, int rows, int cols, int box_rows, CUtensorMap* out);

// ---- rowwise.cu -------------------------------------------------------------------------------------
// GaussianFourierProjection (model.py:85-97): out[b, :] = [sin(x), cos(x)], x = ((t*W)*2)*pi in fp32.
// t = timestep[b], or (float)*step_ptr for every b when step_ptr != NULL (sampling loop, quirk Q3), or (float)b when both are NULL
// (the sampling loop's [T, H] table of steps 0 .. T-1).
// out16 (optional): 16-bit copy in format fmt16 (0 = fp16, 1 = bf16).
int timestep_embed(const float* timestep, const int* step_ptr, const float* W, int B, int H, float* out, void* out16, int fmt16,
                   cudaStream_t s);
// BertEmbeddings (model.py:110-117): out = LN(x @ Wt + b) (+ te[row / L]); Wt is the [fin, H] transpose.  Up to four
// embeddings (jobs) run in one launch.  Rowwise kernels read the fp32 residual stream and may write BOTH an fp32 copy
// (out32: the stream) and a T copy (outT: the operand of the next GEMM); either pointer may be NULL.
struct EmbedJob {
  const float* x;       // [M, fin]
  const float* Wt;      // [fin, H]
  const float* b;       // [H]
  const float* lnw;     // [H]
  const float* lnb;     // [H]
  const float* te;      // [M / L, H] added after the LayerNorm, or NULL
  float* out32;         // [M, H] or NULL
  void* outT;           // [M, H] operand-typed copy or NULL
  int M, fin, L;
  // packed (ragged) mode: output row r is computed from input row src_rows[r] (index into the padded [B * L, fin] input) and takes
  // the timestep features of graph row_graph[r]; NULL = identity / r / L
  const int* src_rows;
  const int* row_graph;
  const int* te_row;  // sampling loop: every row takes te row *te_row (te is then the [T, H] table of the steps), else NULL
  int cta_begin, cta_count;  // filled by embed_ln_multi
};
struct EmbedJobs {
  EmbedJob j[4];
  int n;
  int max_fin;  // filled by embed_ln_multi (smem layout)
  // optional side job: cat_dst = [cat_a (cat_na floats) | cat_b (cat_nb floats)] (stacked key masks)
  float* cat_dst;
  const float* cat_a;
  const float* cat_b;
  int cat_na, cat_nb;
};
template <typename T> int embed_ln_multi(EmbedJobs jobs, float eps, int H, cudaStream_t s);
// out = LayerNorm(in) * w + b
template <typename T>
int layernorm(const float* in, int M, int H, const float* w, const float* b, float eps, float* out32, T* outT, float2* stats, cudaStream_t s);
// (stats[row] = (mean, rstd), optional: a GEMM epilogue can then rebuild LayerNorm(in) as its residual without an fp32 copy)
// SELayer residual update (model.py:61-62):
//   y = affine_first ? LayerNorm(in; lnw, lnb, eps1) : in          (BertSelfOutput.LayerNorm)
//   out = x + gate * (LayerNorm_noaffine(y, 1e-5) * (1 + scale) + shift)
// (shift, scale, gate) = mod[row / mod_div, (chunk0 + {0,1,2}) * H : ...], mod row pitch 6H.
// row_graph (optional, packed mode with graph-level conditioning): row r uses mod row row_graph[r] instead of r / mod_div
// mod_row (optional, sampling loop): every row uses mod row *mod_row (the step's row of a [T, 6H] modulation table)
// in_hi / x_hi (optional, sampling loop): rows r >= split read `in` and `x` from row r - split of these instead
template <typename T>
int ln_modulate(const float* in, int M, int H, bool affine_first, const float* lnw, const float* lnb, float eps1, const float* x,
                const T* mod, int mod_div, int chunk0, float* out32, T* outT, cudaStream_t s, const int* row_graph = nullptr,
                const int* mod_row = nullptr, int split = 0, const float* in_hi = nullptr, const float* x_hi = nullptr);
// AminoAcidPredictor tail (model.py:151-152): logits = LayerNorm(y) @ W2^T + b2  (y is already GELU(dense1))
// dst_rows (optional, packed mode): logits of row r are written to row dst_rows[r] of `logits` (the padded [B * L, F] layout)
template <typename T>
int predictor_tail(const T* y, int M, int H, const float* lnw, const float* lnb, float eps, const float* W2, const float* b2,
                   int F, float* logits, cudaStream_t s, const int* dst_rows = nullptr);
template <typename T> int f32_to_16(const float* in, size_t n, T* out, cudaStream_t s);  // T = bf16 | f16
int transpose_f32(const float* in, int rows, int cols, float* out, cudaStream_t s);  // out[c][r] = in[r][c]
int step_advance(int* step_ptr, cudaStream_t s);                                     // *step_ptr -= 1

// ---- attention.cu -----------------------------------------------------------------------------------
// Packed (ragged) batches: graph b's query rows are rows q_off[b] .. q_off[b] + q_len[b] - 1 of q / out, its key rows k_off[b] .. of
// k / v (device arrays of B ints); Lq / Lk are then the LARGEST query / key length of the batch and Lk_mask the row pitch of
// key_mask (the padded length).  Rows of other graphs that fall into a tile are masked exactly like padding (their probabilities
// underflow to 0), output rows past q_len[b] are not written.  16-bit modes (pipelined tcgen05 kernel) only.
struct AttnPack {
  const int* q_off;
  const int* k_off;
  const int* q_len;
  int q_rows, k_rows;  // total rows of the packed q / k matrices
  int Lk_mask;
};
// kv_div > 1 (B % kv_div == 0): query graph b attends to key graph b / kv_div -- its K / V rows (padded: (b / kv_div) * Lk, packed:
// k_off[b / kv_div]) and its key-mask row.  The sampler's K samples per pocket share one pocket's cross K|V this way.
template <typename T>
int attention(int B, int heads, int Lq, int Lk, const T* q, int ldq, const T* k, int ldk, const T* v, int ldv, const T* dist_emb,
              int P, const float* key_mask, T* out, cudaStream_t s, const AttnPack* pack = nullptr, int kv_div = 1);

// ---- collate.cu ---------------------------------------------------------------------------------------
// LigandBindingSiteDataset.__getitem__ for G ragged complexes (dataset.py:97-129); lengths[g] = (n_lig, n_rec) BEFORE clamping.
int collate(int G, const int* offsets, const uint8_t* lig_mask, const uint8_t* poc_mask, const float* ang, const float* aa, int ext, int L,
            float* lig_ang, float* lig_seq, float* lig_attn, float* rec_ang, float* rec_seq, float* rec_attn, int* lengths, cudaStream_t s);

// ---- attention_tc.cu: tcgen05 attention (S, Q.E^T and P.V on UMMA, accumulators in TMEM) ------------------------------
template <typename T>
int attention_tc(int B, int heads, int Lq, int Lk, const T* q, int ldq, const T* k, int ldk, const T* v, int ldv, const T* dist_emb,
                 int P, const float* key_mask, T* out, cudaStream_t s);
extern unsigned long long* g_attn_trace;  // debug timeline buffer of the pipelined kernel (NULL = off)
// ---- attention_pipe.cu: persistent, warp-specialised version (TMA / MMA / softmax roles pipelined over work items) -----
template <typename T>
int attention_pipe(int B, int heads, int Lq, int Lk, const T* q, int ldq, const T* k, int ldk, const T* v, int ldv, const T* dist_emb,
                   int P, const float* key_mask, T* out, cudaStream_t s, const AttnPack* pack = nullptr, int kv_div = 1);
// ---- attention_bwd_pipe.cu: backward of the attention core on tcgen05 (Lq, Lk <= 128; dE += gradient of the distance embedding) ----
bool attention_bwd_pipe_usable(int Lq, int Lk, const void* dist_emb, float p_drop);
template <typename T>
int attention_bwd_pipe(int B, int heads, int Lq, int Lk, const T* q, int ldq, const T* k, int ldk, const T* v, int ldv, const T* dist_emb, int P,
                       const float* key_mask, DropSpec dr, const T* dout, T* dq, int lddq, T* dk, int lddk, T* dv, int lddv, float* dE, cudaStream_t s,
                       const uint32_t* keep_in = nullptr);
// the same kernel with the training-mode attention-probability dropout applied to P (masks: DropSpec / Philox, philox.cuh); Lk % 4 == 0
template <typename T>
int attention_pipe_dropout(int B, int heads, int Lq, int Lk, const T* q, int ldq, const T* k, int ldk, const T* v, int ldv, const T* dist_emb,
                           int P, const float* key_mask, DropSpec dr, T* out, cudaStream_t s, uint32_t* keep_out = nullptr);
// keep_out / keep_in: [B * heads][128 rows][4] words, bit j of word kc = "key 32 kc + j of that query is kept" (Lq, Lk <= 128); written by the
// forward, read by attention_bwd_pipe instead of regenerating the Philox stream


// ---- reverse_step.cu --------------------------------------------------------------------------------
// step_ptr != NULL: tables/noise are indexed by *step_ptr (entry stride 1200 / N*20) and the launch is a
// no-op when *step_ptr == 0 (last step returns the raw logits, sample.py:147-148).
int reverse_step(const float* q_tables, int n_tab, int B, int L, const float* x_t, const float* logits, int diverse,
                 const float* noise_E, uint64_t seed, uint64_t graph_id0, uint32_t step, const int* step_ptr, float* x_s,
                 uint8_t* idx_out, cudaStream_t s, int* advance = nullptr, const uint64_t* rng = nullptr);
// advance != NULL (with step_ptr): advance[0] is a zeroed arrival counter; the last CTA to have read *step_ptr decrements it
// (replaces a separate step_advance launch in the sampling loop)
// rng != NULL: device pointer to (seed, graph_id0), overriding the by-value arguments (kernel parameters are frozen into a captured
// CUDA graph; device memory is not, so one cached graph serves calls with different seeds / graph offsets).
// In-place contract: x_s may alias x_t (the loop does that) -- every thread reads its own 20-float row completely before writing it.
int apply_aa_noise(const float* qtb, int B, int L, const float* x0, const float* noise_E, uint64_t seed, uint64_t graph_id0,
                   uint32_t step, float* x_t, uint8_t* idx_out, cudaStream_t s);
int philox_u32(uint64_t seed, uint64_t graph_id0, uint32_t step, int B, int L, uint32_t* out, cudaStream_t s);

// ---- decode_loss.cu ---------------------------------------------------------------------------------
// sample.py:208-224: pred_idx / true_idx [B*L] = argmax rows; counts [B,2] = (#masked matches, #masked)
int decode_sequences(int B, int L, const float* final_seq, const float* true_seq, const float* mask, uint8_t* pred_idx, uint8_t* true_idx,
                     int* counts, cudaStream_t s);
// model.py:313-345 + utils.py:132-161: the ten reduction terms documented at seqdiff_loss_terms (include/seqdiff_b200.h).
// The per-CTA partials live in stream-ordered scratch (cudaMallocAsync / cudaFreeAsync on `s`).
int loss_terms(int N, const float* logits, const float* x0, const float* x_t, const float* mask, double* terms, cudaStream_t s,
               double* scratch = nullptr);  // scratch (optional): loss_terms_scratch_bytes() of caller-owned, stream-private memory
size_t loss_terms_scratch_bytes();

// ---- gauss_step.cu ----------------------------------------------------------------------------------
// Gaussian reverse step + angle wrap of the structure model (structure_model/sample.py:92-101,139-141) on B graphs of
// per_graph = L * F elements.  coef [T,4] = (1/sqrt(alpha), beta, sqrt(1 - alphabar), sqrt(posterior_variance)) per step.
// noise: N(0,1) values (one [B*per_graph] block; with step_ptr a [T, B*per_graph] table indexed by the step) or NULL ->
// in-kernel Philox + Box-Muller.  step_ptr / advance as in reverse_step().  steps_out (optional) [T, B*per_graph]: the result
// is also stored at entry T-1-step (the reference's per-step history).  wrap = false: p_sample's un-wrapped value.
int gauss_step(const float* coef, int T, int B, int per_graph, const float* x_t, const float* model_out, const float* noise, uint64_t seed,
               uint64_t graph_id0, int step, const int* step_ptr, float* x_out, float* steps_out, cudaStream_t s, int* advance = nullptr, bool wrap = true,
               const uint64_t* rng = nullptr);  // rng / in-place (x_out == x_t) as in reverse_step()

// ---- train_kernels.cu / attention_train.cu: the training step (reference model.py:313-367 under autograd) ------------
// out[c][r] = in[r][c] for row-major [rows, cols]; colsum (optional, fp32 [cols]) += column sums (bias gradients); out may be NULL.
// pitch (default rows): row pitch of `out` in elements, rows <= pitch < rows + 64; columns rows..pitch-1 are written as zeros (the
// contraction dimension of the weight-gradient GEMM must be a multiple of 8 elements for TMA)
template <typename T> int colsum_add(const T* in, int rows, int cols, float* colsum, cudaStream_t s);  // colsum[c] += sum_r in[r, c]
template <typename T> int transpose_colsum(const T* in, int rows, int cols, T* out, float* colsum, cudaStream_t s, int pitch = 0);
template <typename T> int transpose_cast(const float* in, int rows, int cols, T* out, cudaStream_t s);  // fp32 [r,c] -> T [c,r]
// a = dropout(act(z)), kind 1 = erf-GELU, 2 = SiLU;  dz = da * keep * act'(z)
template <typename T> int act_fwd(const T* z, size_t n, int kind, DropSpec dr, T* a, cudaStream_t s);
template <typename T, typename TG> int act_bwd(const TG* da, const T* z, size_t n, int kind, DropSpec dr, T* dz, cudaStream_t s);
int dropout_add(float* d, const float* resid, size_t n, DropSpec dr, cudaStream_t s);           // d = dropout(d) + resid (resid may be NULL)
template <typename T> int grad_cast(const float* g, size_t n, DropSpec dr, T* out, cudaStream_t s);  // out = T(g * keep)
// d <- o = dropout(d) + resid;  out32 / outT (either optional) = LayerNorm(o) * w + b: dropout_add + layernorm in one pass;
// keep_bits (optional) [M, H / 8] bytes: the mask, for layernorm_bwd_cast
template <typename T>
int dropout_add_layernorm(float* d, const float* resid, DropSpec dr, int M, int H, const float* w, const float* b, float eps, float* out32, T* outT,
                          uint8_t* keep_bits, cudaStream_t s);
// h = LN(o) * gamma + beta:  d_o = LN-backward(dh); dgamma / dbeta += row sums (atomic, fp32 [H])
int layernorm_bwd(const float* dh, const float* o, int M, int H, const float* gamma, float eps, float* d_o, float* dgamma, float* dbeta,
                  cudaStream_t s);
// the same, and in the same pass: gT = T(d_o * keep) (the 16-bit dY operand of the Linear that produced o) and dbias += column sums of gT;
// keep_bits (optional): the mask as dropout_add_layernorm() stored it, else regenerated from `dr`
template <typename T>
int layernorm_bwd_cast(const float* dh, const float* o, int M, int H, const float* gamma, float eps, float* d_o, float* dgamma, float* dbeta,
                       DropSpec dr, const uint8_t* keep_bits, T* gT, float* dbias, cudaStream_t s);
// backward of ln_modulate(): din = gradient of `in`; sum_out (optional) = din + dout; d(shift, scale, gate) -> dmodT rows (mod_div == 1)
// or atomically into dmod32 [M / mod_div, 6H]; dgamma / dbeta of the affine LayerNorm when affine_first
template <typename T>
int ln_modulate_bwd(const float* dout, const float* in, int M, int H, bool affine_first, const float* lnw, const float* lnb, float eps1,
                    const T* mod, int mod_div, int chunk0, float* din, float* sum_out, T* dmodT, float* dmod32, float* dgamma, float* dbeta,
                    cudaStream_t s);
int embed_bwd(const float* dout, const float* x, int M, int fin, int H, const float* Wt, const float* b, const float* gamma, float eps, DropSpec dr,
              float* dW, float* db, float* dgamma, float* dbeta, cudaStream_t s);
template <typename T>
int predictor_tail_bwd(const float* dlogits, const T* y, int M, int H, const float* gamma, const float* beta, float eps, const float* W2, int F,
                       float* dy, float* dW2, float* db2, float* dgamma, float* dbeta, cudaStream_t s);
// d(total loss)/d(logits) with total = CE_mean(noised) + elbo_loss(noised); terms = output of loss_terms() (terms[1] = #noised)
int loss_bwd(int N, const float* logits, const float* x0, const float* x_t, const double* terms, float* dlogits, cudaStream_t s);
// clip_grad_norm_(max_norm) + AdamW over the flat buffers; d_w / d_off: device tables (master pointers, flat offsets [n + 1]);
// grad_scale folds the 1 / world of the gradient average; d_scratch: 2 * #SM + 8 doubles; norm_out (optional): the pre-clip norm
int adamw_step(float* const* d_w, const int64_t* d_off, int n_slots, size_t total, const float* g, float* m, float* v, float grad_scale,
               float max_norm, float lr, float beta1, float beta2, float eps, float wd, int step, double* d_scratch, float* norm_out, cudaStream_t s);
// attention with probability dropout (forward) and its backward; SIMT fp32 arithmetic, Lk <= 128.  dq / dk / dv carry their own
// row strides (they are slices of the fused [M, 3H] / [M, layers * 2H] gradient tensors); dE [2P-1, 64] fp32 is accumulated.
template <typename T>
int attention_train_fwd(int B, int heads, int Lq, int Lk, const T* q, int ldq, const T* k, int ldk, const T* v, int ldv, const T* dist_emb, int P,
                        const float* key_mask, DropSpec dr, T* out, cudaStream_t s);
template <typename T>
int attention_bwd(int B, int heads, int Lq, int Lk, const T* q, int ldq, const T* k, int ldk, const T* v, int ldv, const T* dist_emb, int P,
                  const float* key_mask, DropSpec dr, const T* dout, T* dq, int lddq, T* dk, int lddk, T* dv, int lddv, float* dE, cudaStream_t s);

// attention_train_tc.cu: the same two operations on warp-level tensor-core MMAs (16-bit modes; the SIMT kernels above stay the fp32
// parity path and the reference these are tested against)
template <typename T>
int attention_train_fwd_tc(int B, int heads, int Lq, int Lk, const T* q, int ldq, const T* k, int ldk, const T* v, int ldv, const T* dist_emb, int P,
                           const float* key_mask, DropSpec dr, T* out, cudaStream_t s);
template <typename T>
int attention_bwd_tc(int B, int heads, int Lq, int Lk, const T* q, int ldq, const T* k, int ldk, const T* v, int ldv, const T* dist_emb, int P,
                     const float* key_mask, DropSpec dr, const T* dout, T* dq, int lddq, T* dk, int lddk, T* dv, int lddv, float* dE, cudaStream_t s);

}  // namespace seqdiff
