// model.cuh -- the seqdiff model handle (opaque `seqdiff_model_t` of the C ABI).
#pragma once
#include <map>
#include <string>
#include <vector>

#include "kernels.h"

namespace seqdiff {

// one logical matrix in the three storage formats (16-bit copies made by finalize())
struct Wt {
  const float* f = nullptr;
  const bf16* h = nullptr;
  const f16* g = nullptr;
  const void* t = nullptr;  // training only: the TRANSPOSED matrix [in, out] in the training precision's operand type (dgrad GEMMs)
  int64_t rows = 0, cols = 0;  // [out, in]
};

struct AttnW {
  Wt qkv;  // [3H,H] rows = query | key | value  (self-attention only)
  const float* qkv_b = nullptr;
  Wt E;  // distance_embedding [2P-1,64] or null
  Wt out;
  const float *out_b = nullptr, *ln_w = nullptr, *ln_b = nullptr;
};
struct SEW {  // SELayer, model.py:26-66
  Wt ada0, ada2, m0, m3;
  const float *ada0_b = nullptr, *ada2_b = nullptr, *m0_b = nullptr, *m3_b = nullptr;
  AttnW attn;
};
struct LayerW {  // HF BertLayer; the cross-attention members stay empty for an encoder layer (structure model)
  AttnW self;
  Wt cq, cout, inter, outd;
  const float *cq_b = nullptr, *cout_b = nullptr, *cln_w = nullptr, *cln_b = nullptr;
  const float *inter_b = nullptr, *outd_b = nullptr, *oln_w = nullptr, *oln_b = nullptr;
};
struct EmbW {  // BertEmbeddings, model.py:99-117
  const float *Wt_ = nullptr, *b = nullptr, *ln_w = nullptr, *ln_b = nullptr;
  int fin = 0;
};

struct RawTensor {
  float* ptr = nullptr;
  int64_t numel = 0;
  bool set = false;
};

struct ParamSlot {  // one trainable tensor: fp32 master + its place in the flat gradient / AdamW-state buffers
  std::string name;
  float* w = nullptr;
  int64_t numel = 0, off = 0;
};

// arguments of one training step (forward + loss + backward): reference model.py:313-367
struct TrainArgs {
  int precision, B, Ll, Lr;
  const float *t_norm, *x_t, *x0, *lig_angle, *lig_mask, *rec_seq, *rec_angle, *rec_mask;
  float p_hidden, p_attn;
  uint64_t seed;
  uint32_t step;
  float* grads;      // flat fp32 [train_param_count()], overwritten
  double* terms;     // [10] loss terms (seqdiff_loss_terms layout)
  float* logits_out; // optional [B, Ll, feature_size]
};

// arguments of one training step of the structure model (forward + wrapped smooth-L1 loss + backward)
struct StructTrainArgs {
  int precision, B, Ll, Lr;
  const float *t, *corrupted, *known_noise, *lig_mask, *rec_seq, *rec_angle, *rec_mask;
  float p_hidden, p_attn;
  uint64_t seed;
  uint32_t step;
  float* grads;     // flat fp32 [train_param_count()], overwritten
  double* terms;    // [feature_size + 1]: per-feature loss sums, then the number of valid ligand positions
  float* pred_out;  // optional [B, Ll, feature_size]
};

struct Segment {  // a run of graphs sharing one padded length inside a token matrix
  int row0, B, L;
  const float* mask;
};

int profile_begin(cudaStream_t s);
int profile_end(char* tags, int tag_stride, float* ms, int* counts, int cap);

// Ragged packing of a sampling batch (DESIGN.md "Ragged batches"): only the valid prefix of every graph is computed.  Token rows of
// graph b occupy rows [off[b], off[b] + len[b]) of every [rows, H] matrix; all index arrays live in one device block.  A sampling
// of K samples per pocket has B = P * K ligand graphs and P receptor graphs (sample b reads pocket b / K).
struct PackInfo {
  int B = 0, P = 0, Ml = 0, Mr = 0;  // ligand / receptor graphs, packed ligand / receptor row counts
  int max_l = 0, max_r = 0;       // largest ligand / receptor length
  const int* src_l = nullptr;     // [Ml] packed ligand row -> padded row index b * Ll + l
  const int* src_r = nullptr;     // [Mr]
  const int* graph = nullptr;     // [Ml + Mr] graph of a stacked row (receptor rows: the pocket)
  const int* off_l = nullptr;     // [B] first ligand row of graph b
  const int* off_r = nullptr;     // [P] first receptor row of pocket p, relative to the receptor block
  const int* len_l = nullptr;     // [B]
  const int* len_r = nullptr;     // [P]
  const int* off_cat = nullptr;   // [B + P] ligand offsets, then receptor offsets + Ml (stacked matrix)
  const int* len_cat = nullptr;   // [B + P]
  uint64_t hash = 0;              // of K, lig_padded and the length vectors (part of the CUDA-graph key)
  // Receptor-only pack (the padded sampling loop): the ligand rows keep their padded layout -- every ligand length is Ll, so
  // Ml = B * Ll, src_l is the identity and off_l[b] = b * Ll -- and only the receptor rows are packed.  No output reads a padded
  // receptor row (DESIGN.md section 9), so the result is the padded computation's at every position, padded ones included.
  bool lig_padded = false;
};

// What the sequence model's sampling loop computes once per sampling instead of once per step (Model::sample).  Every graph of the
// batch shares the step index and x_t is the only other input that changes between steps, so the receptor embedding, the receptor
// half of ligand_feature_emb's attention sublayer (its input is the receptor embedding alone), the timestep features and
// decoder_normalize's modulation (a function of the timestep features alone) are the same at every step.  The buffers are carved
// from the handle's samp_inv block; receptor rows are [Mr, H] in the row order of the step's token matrix (packed or padded), one
// set per pocket: the K samples of a pocket share them.
struct LoopInv {
  int rows = 0;          // table capacity in steps (>= T of the sampling)
  float* xr = nullptr;   // [Mr, H] receptor embedding, fp32 stream
  void* xrT = nullptr;   // [Mr, H] its operand copy (== xr in fp32 mode)
  float* o = nullptr;    // [Mr, H] receptor rows of ligand_feature_emb's attention output (dense + residual, before its LayerNorm)
  float* te = nullptr;   // [rows, H] timestep features of step i in row i
  void* teT = nullptr;   // [rows, H] operand copy (== te in fp32 mode)
  void* u = nullptr;     // [rows, H] SiLU(adaLN_modulation.0) of decoder_normalize (scratch of the table)
  void* mod = nullptr;   // [rows, 6H] decoder_normalize's modulation (shift, scale, gate) x 2 of step i in row i
};

enum Arch { kArchSequence = 0, kArchStructure = 1 };

struct Model {
  seqdiff_config_t cfg{};
  int arch = kArchSequence;  // which reference module tree the handle holds (sequence_model/model.py | structure_model/model.py)
  int device = 0;
  bool finalized = false;
  std::map<std::string, RawTensor> raw;  // reference state_dict key -> fp32 device tensor
  std::vector<void*> allocs;         // raw tensors + small state (life of the handle)
  std::vector<void*> packed_allocs;  // fused / bf16 copies made by finalize()
  bool packing = false;

  EmbW lig_seq, lig_ang, rec_seq, rec_ang;
  SEW se_lig, se_dec;
  std::vector<LayerW> layers;      // decoder
  std::vector<LayerW> enc_layers;  // structure model only: the 12-layer receptor encoder (self-attention + FFN)
  Wt ckv_all;  // all layers' cross key|value weights stacked: [layers*2H, H]
  const float* ckv_all_b = nullptr;
  Wt p1;
  const float *p1_b = nullptr, *p_ln_w = nullptr, *p_ln_b = nullptr, *p2_w = nullptr, *p2_b = nullptr, *ts_W = nullptr;

  // workspace (grow-only)
  uint8_t* ws = nullptr;
  size_t ws_bytes = 0;

  // sampling-loop state
  int* d_step = nullptr;
  float* d_tables = nullptr;
  size_t tables_cap = 0;
  uint8_t* samp_in = nullptr;  // persistent copies of the loop inputs + x_t + logits
  size_t samp_in_bytes = 0;
  uint8_t* samp_inv = nullptr;  // the LoopInv buffers (grow-only)
  size_t samp_inv_bytes = 0;
  LoopInv inv;
  cudaGraphExec_t graph_exec = nullptr;
  int graph_kernels = 0;
  cudaStream_t loop_stream = nullptr;  // private stream: graphs cannot be captured on the legacy default stream
  cudaEvent_t ev_in = nullptr, ev_out = nullptr;
  struct GraphKey {
    int precision = -1, B = 0, K = 0, Ll = 0, Lr = 0, diverse = 0;
    const float* noise = nullptr;
    const void* ws_ptr = nullptr;
    const void* in_ptr = nullptr;
    const void* tab_ptr = nullptr;
    const void* aux_ptr = nullptr;
    const void* inv_ptr = nullptr;
    int inv_rows = 0;  // with B, K, Lr and the precision: the layout of the LoopInv buffers
    int T = 0;
    uint64_t pack_hash = 0;
    bool operator==(const GraphKey& o) const {
      return pack_hash == o.pack_hash && aux_ptr == o.aux_ptr && T == o.T && precision == o.precision && B == o.B && K == o.K && Ll == o.Ll && Lr == o.Lr && diverse == o.diverse && noise == o.noise &&
             ws_ptr == o.ws_ptr && in_ptr == o.in_ptr && tab_ptr == o.tab_ptr && inv_ptr == o.inv_ptr && inv_rows == o.inv_rows;
    }
  } graph_key;

  ~Model();
  int init(const seqdiff_config_t& c, int dev, int arch_ = kArchSequence);
  int set_tensor(const char* name, const float* data, int64_t numel, cudaStream_t s);
  int finalize(cudaStream_t s);
  // inv != NULL (sampling loop, with step_ptr): the step reads what loop_invariants_t() left in `inv` instead of recomputing it;
  // rec_seq is not read then.  K > 1 (with inv only): the receptor inputs hold B / K pockets and ligand graph b uses pocket b / K.
  int forward(int precision, int B, int Ll, int Lr, const float* timestep, const int* step_ptr, const float* x_t,
              const float* lig_angle, const float* lig_mask, const float* rec_seq, const float* rec_angle, const float* rec_mask,
              float* logits, cudaStream_t s, const PackInfo* pk = nullptr, const LoopInv* inv = nullptr, int K = 1);
  // P pockets x K samples per pocket: ligand inputs / x_T / final_out hold B = P * K graphs (sample j of pocket p is graph
  // p * K + j), receptor inputs hold P.  flags bit 0: ragged packing (valid positions bit-identical to the padded computation;
  // padded positions of final_out are 0)
  int sample(int precision, int P, int K, int Ll, int Lr, int T, const float* q_tables, const float* x_T, const float* lig_angle,
             const float* lig_mask, const float* rec_seq, const float* rec_angle, const float* rec_mask, int diverse,
             const float* noise_E, uint64_t seed, uint64_t gid0, float* final_out, cudaStream_t s, int flags = 0);
  // The same loop scoring given sequences x0 (P * K graphs, one-hot at the valid positions) under the sampler's variational bound:
  // T x (q-sample x_t ~ q(x_t | x0) with the step's Qtb -> forward -> vlb_terms), replayed from its own captured graph (score_exec),
  // so that alternating sample / score calls on one handle keep both graphs.  terms_out [P * K, Ll, 2] fp64 (device or host):
  // per residue (prior-free bound terms summed over the steps, cross-entropy summed over the steps); 0 at masked positions.
  int score(int precision, int P, int K, int Ll, int Lr, int T, const float* q_tables, const float* x0, const float* lig_angle,
            const float* lig_mask, const float* rec_seq, const float* rec_angle, const float* rec_mask, const float* noise_E,
            uint64_t seed, uint64_t gid0, double* terms_out, cudaStream_t s, int flags = 0);
  uint8_t* score_in = nullptr;  // x0 + the fp64 sums of the scoring loop (grow-only; a structure handle adds the q-sample table)
  size_t score_in_bytes = 0;
  cudaGraphExec_t score_exec = nullptr;
  int score_kernels = 0;
  GraphKey score_key;
  // what sample() and score() share: the loop's buffers in the persistent input block, the packing and the step-graph key
  struct LoopIO {
    float *x_cur, *logits, *c_lang, *c_lmask, *c_rseq, *c_rang, *c_rmask;
    float* x0 = nullptr;     // score only: the scored sequences
    double* acc = nullptr;   // score only: [B * Ll, 2] fp64 sums (zeroed by loop_setup)
    const PackInfo* pk = nullptr;
    long long rows = 0;      // token rows of a step
    GraphKey key;
  };
  // Private stream ordered after `caller`, persistent copies of the inputs (x_in -> x_cur for sampling, -> x0 for scoring), the step
  // tables, the workspace, the packing (flags bit 0) and the LoopInv of this call.  Returns the loop stream in *ls.
  int loop_setup(int precision, int P, int K, int Ll, int Lr, int T, const float* q_tables, const float* x_in, const float* lig_angle,
                 const float* lig_mask, const float* rec_seq, const float* rec_angle, const float* rec_mask, cudaStream_t caller, int flags,
                 bool scoring, LoopIO* io, cudaStream_t* ls);
  // (Re)captures `step` into `exec` unless `key` matches the cached key (dry run of `fwd` first), then arms the step counter at T - 1
  // with the Philox key (seed, gid0) and replays the graph T times on s.
  template <typename Fwd, typename Step>
  int replay_loop(cudaGraphExec_t& exec, GraphKey& cached, int& kernels, const GraphKey& key, int T, uint64_t seed, uint64_t gid0, cudaStream_t s,
                  const Fwd& fwd, const Step& step);
  int* d_pack = nullptr;  // device block behind PackInfo (grow-only)
  size_t pack_cap = 0;
  PackInfo pack;
  // lig_padded: the receptor-only pack (PackInfo::lig_padded); lig_mask is not read then
  int build_pack(int B, int K, int Ll, int Lr, const float* lig_mask, const float* rec_mask, cudaStream_t s, bool* usable,
                 bool lig_padded = false);

  // ---- training (train.cu) ------------------------------------------------------------------------------------------
  std::vector<ParamSlot> slots;            // trainable tensors in flat-buffer order (fused groups contiguous)
  std::map<std::string, int> slot_of;
  int64_t train_total = 0;
  std::vector<int64_t> grad_bucket_bounds;  // flat offsets [n+1]: the backward pass finishes bucket n-1 first, bucket 0 last
  std::vector<cudaEvent_t> bucket_events;   // caller-owned; event k is recorded on the training stream once bucket k is final
  int train_prec = -1;                     // precision the transposed operand copies (Wt::t) were built for; -1 = none
  bool repack_reuse = false;               // finalize() after an optimizer step: re-fill the packed buffers in place
  size_t packed_cursor = 0;
  // The packing operations of the last full finalize(), recorded so that the refresh after an optimizer step is three batched
  // launches (copies, conversions, transposes) over device-resident chunk tables instead of ~270 small ones.
  struct RpCopy { float* dst; const float* src; int64_t n; };
  struct RpConv { const float* src; void* h; void* g; int64_t n; };
  struct RpTrans { const float* src; void* dst; int rows, cols; };
  std::vector<RpCopy> rp_copy;
  std::vector<RpConv> rp_conv;
  std::vector<RpTrans> rp_trans, rp_trans_f32;
  void* d_rp_tables = nullptr;             // chunk tables of the three batched kernels (built on first use)
  int rp_n_copy = 0, rp_n_conv = 0, rp_n_trans = 0, rp_n_trans_f32 = 0, rp_table_prec = -2;
  int repack_fast(cudaStream_t s);
  float** d_slot_w = nullptr;
  int64_t* d_slot_off = nullptr;
  double* d_opt_scratch = nullptr;
  float* d_zero_bias = nullptr;
  uint8_t* tws = nullptr;                  // training workspace (tape + backward buffers), grow-only
  size_t tws_bytes = 0;
  int build_slots();
  int64_t train_param_count();
  int train_prologue(int precision, int B, int Ll, int Lr, float p_hidden, float p_attn, cudaStream_t s);
  int train_step(const TrainArgs& a, cudaStream_t s);
  int struct_train_step(const StructTrainArgs& a, cudaStream_t s);
  int adamw(const float* grads, float* m, float* v, float grad_scale, float max_norm, float lr, float beta1, float beta2, float eps, float wd,
            int step, float* norm_out, cudaStream_t s);
  int get_tensor(const char* name, float* out, int64_t numel, cudaStream_t s);
  template <typename T> int train_t(int wfmt, const TrainArgs& a, cudaStream_t s);
  template <typename T> int struct_train_t(const StructTrainArgs& a, cudaStream_t s);

  // structure_model/model.py:180-215.  phases: bit 0 = run the receptor branch, bit 1 = the ligand branch.  The receptor branch (embeddings,
  // receptor_emb, encoder, all decoder layers' cross K|V) depends on neither the timestep nor the ligand, so the sampling loop runs it
  // once and keeps the K|V block.
  // pk (16-bit modes, sampling loop): ragged packing (build_pack(B, K, ...)).  K > 1 (sampling loop): the receptor inputs hold B / K
  // pockets, the receptor branch runs over them once, and ligand graph b cross-attends to pocket b / K.
  int struct_forward(int precision, int B, int Ll, int Lr, const float* timestep, const int* step_ptr, const float* noised_angles,
                     const float* lig_mask, const float* rec_seq, const float* rec_angle, const float* rec_mask, float* out, int phases,
                     cudaStream_t s, const PackInfo* pk = nullptr, int K = 1);
  // structure_model/sample.py:104-144 (STEP = 1): T x (forward, Gaussian reverse step, angle wrap) from one captured graph.
  // P pockets x K samples per pocket: ligand inputs / x_T / noise / steps_out / final_out hold B = P * K graphs (sample j of pocket p
  // is graph p * K + j), receptor inputs hold P.
  // flags bit 0: ragged packing (valid positions bit-identical to the padded loop; padded positions of steps_out / final_out are 0)
  int struct_sample(int precision, int P, int K, int Ll, int Lr, int T, const float* coef_steps, const float* x_T, const float* lig_mask,
                    const float* rec_seq, const float* rec_angle, const float* rec_mask, const float* noise_steps, uint64_t seed,
                    uint64_t gid0, float* steps_out, float* final_out, cudaStream_t s, int flags = 0);
  // The same loop scoring given backbones x0 (P * K graphs) under the structure model's training objective: T x (q-sample x_k from x0
  // at step k -> ligand branch at timestep k -> terms += h(wrap(eps_k - pred))), replayed from its own captured graph (score_exec /
  // score_key, which a structure handle does not otherwise use), so that alternating sample / score calls keep both graphs.
  // qs_steps [T, 2] = (sqrt(alphabar), sqrt(1 - alphabar)); terms_out [P * K, Ll, F] fp64 (device or host): per element, the sum over
  // the steps of the wrapped smooth-L1; 0 at masked positions.  flags bit 0: ragged packing (bit-identical terms at valid positions).
  int struct_score(int precision, int P, int K, int Ll, int Lr, int T, const float* qs_steps, const float* x0, const float* lig_mask,
                   const float* rec_seq, const float* rec_angle, const float* rec_mask, const float* noise_steps, uint64_t seed,
                   uint64_t gid0, double* terms_out, cudaStream_t s, int flags = 0);
  // what struct_sample() and struct_score() share: the loop's buffers in the persistent input block, the packing and the step-graph key
  struct StructIO {
    float *x_cur, *mout, *c_lmask, *c_rseq, *c_rang, *c_rmask;
    float* x0 = nullptr;    // score only, in score_in: the scored backbones ...
    double* acc = nullptr;  // ... the [B * Ll, F] fp64 sums (zeroed by struct_loop_setup) ...
    float* qs = nullptr;    // ... and, last (its size depends on T), the [T, 2] q-sample table
    const PackInfo* pk = nullptr;
    GraphKey key;
  };
  // Private stream ordered after `caller`, persistent copies of the inputs (x_in -> x_cur, and -> x0 for scoring), the step table
  // (sampling: coef -> d_tables; scoring: qs -> the score block), the workspace and the packing (flags bit 0).  Returns the stream in *ls.
  int struct_loop_setup(int precision, int P, int K, int Ll, int Lr, int T, const float* table, const float* x_in, const float* lig_mask,
                        const float* rec_seq, const float* rec_angle, const float* rec_mask, cudaStream_t caller, int flags, bool scoring,
                        StructIO* io, cudaStream_t* ls);
  // Arms the step counter at T - 1 with the Philox key (seed, gid0), runs the receptor branch eagerly (with the ligand branch as the
  // un-captured dry run when `step` has to be (re)captured into `exec`, i.e. unless `key` matches the cached key), replays T times.
  template <typename Step>
  int struct_replay(cudaGraphExec_t& exec, GraphKey& cached, int& kernels, const GraphKey& key, int precision, int K, int Ll, int Lr, int T,
                    uint64_t seed, uint64_t gid0, const StructIO& io, cudaStream_t s, const Step& step);

 public:
  void* dalloc(size_t bytes);
  size_t struct_workspace_need(int precision, int B, int Ll, int Lr, int K = 1) const;
  template <typename T>
  int struct_forward_t(int wfmt, int B, int Ll, int Lr, const float* timestep, const int* step_ptr, const float* noised_angles,
                       const float* lig_mask, const float* rec_seq, const float* rec_angle, const float* rec_mask, float* out, int phases,
                       cudaStream_t s, const PackInfo* pk, int K);
  size_t workspace_need(int precision, int B, int Ll, int Lr) const;
  int ensure_workspace(size_t bytes);
  template <typename T>
  int forward_t(int wfmt, int B, int Ll, int Lr, const float* timestep, const int* step_ptr, const float* x_t, const float* lig_angle,
                const float* lig_mask, const float* rec_seq, const float* rec_angle, const float* rec_mask, float* logits,
                cudaStream_t s, const PackInfo* pk, const LoopInv* inv, int K);
  // fills `inv` for a sampling of T_ <= inv.rows steps (Model::sample); scratch from the forward's workspace
  template <typename T>
  int loop_invariants_t(int wfmt, int B, int K, int Ll, int Lr, int T_, const float* rec_seq, const float* rec_mask, const LoopInv& inv,
                        cudaStream_t s, const PackInfo* pk);
};

}  // namespace seqdiff
