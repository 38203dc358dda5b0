// model.cu -- host-side orchestration of the denoiser forward (sequence_model/model.py:200-237) and of
// the reverse-diffusion loop (sequence_model/sample.py:192-207) on top of the kernels in this directory.
//
// Data layout in HBM.  Tokens are rows: a padded batch [B, L, H] is a row-major [B*L, H] matrix; the
// ligand and the receptor batches are stacked into ONE matrix [B*L_lig + B*L_rec, H] because the
// reference runs both through the same SELayer weights (quirk Q1, model.py:221), so every Linear of
// that block is one GEMM over all tokens.  The six cross-attention K|V projections of the decoder act on
// the same receptor features, so they are one GEMM against the stacked [6*2H, H] weight.  Q|K|V of every
// self-attention are one GEMM against the stacked [3H, H] weight.  Activations are bf16 (product) or
// fp32 (parity mode); LayerNorm statistics, softmax, biases and logits are always fp32.
#include "model.cuh"

#include <mutex>
#include <vector>

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <type_traits>

namespace seqdiff {

static thread_local std::string g_err;
void set_error(const std::string& msg) { g_err = msg; }
const char* last_error() { return g_err.c_str(); }
std::atomic<uint64_t> g_launches{0};

// ---- event profiler: one CUDA event behind every tagged launch; durations = gaps between consecutive events of
// one stream (kernels of a stream run back to back).  Used by bench.py for the live roofline numbers.
bool g_profiling = false;
struct ProfMark { const char* tag; cudaEvent_t ev; cudaStream_t s; };
static std::vector<ProfMark> g_marks;
void profile_mark(const char* tag, cudaStream_t s) {
  cudaStreamCaptureStatus st = cudaStreamCaptureStatusNone;
  if (cudaStreamIsCapturing(s, &st) != cudaSuccess || st != cudaStreamCaptureStatusNone) return;  // not inside graph capture
  cudaEvent_t ev;
  if (cudaEventCreate(&ev) != cudaSuccess) return;
  cudaEventRecord(ev, s);
  g_marks.push_back({tag, ev, s});
}
int profile_begin(cudaStream_t s) {
  for (auto& m : g_marks) cudaEventDestroy(m.ev);
  g_marks.clear();
  g_profiling = true;
  profile_mark("__begin__", s);
  return SEQDIFF_OK;
}
// writes up to `cap` records "tag" / total ms / launch count (aggregated per tag); returns the number of tags
int profile_end(char* tags, int tag_stride, float* ms, int* counts, int cap) {
  g_profiling = false;
  if (cudaDeviceSynchronize() != cudaSuccess) return -1;
  std::map<std::string, std::pair<double, int>> agg;
  std::map<cudaStream_t, cudaEvent_t> prev;
  for (auto& m : g_marks) {
    auto it = prev.find(m.s);
    if (it != prev.end() && std::string(m.tag) != "__begin__") {
      float t = 0.f;
      if (cudaEventElapsedTime(&t, it->second, m.ev) == cudaSuccess) {
        auto& a = agg[m.tag];
        a.first += t;
        a.second += 1;
      }
    }
    prev[m.s] = m.ev;
  }
  int n = 0;
  for (auto& kv : agg) {
    if (n >= cap) break;
    std::snprintf(tags + static_cast<size_t>(n) * tag_stride, tag_stride, "%s", kv.first.c_str());
    ms[n] = static_cast<float>(kv.second.first);
    counts[n] = kv.second.second;
    ++n;
  }
  for (auto& m : g_marks) cudaEventDestroy(m.ev);
  g_marks.clear();
  return n;
}

// Programmatic dependent launch.  Modes: 0 off, 1 every launch, 3 only heavy successors, i.e. kernels with >= 64 KB of shared memory
// (the GEMM and attention kernels).  Chosen per call from the measured behaviour on B200 inside the replayed CUDA graph --
//   structure model (M = 4096 steps, 146 kernels of ~10 us): every launch, +2.5 .. 2.7 % (profiles/struct_bench_r01.json);
//   sequence path, <= 2048 stacked token rows (grids of a few CTAs): every launch, B = 1 685 -> 616 us per step (profiles/pdl_small_r02.log);
//   sequence path, <= 32768 rows (cfg 2: 16384 padded, ~7000 packed): heavy successors only, +1.1 % padded / +5.3 % packed; every launch
//     costs 3 % there (the early-launched light kernels take registers next to the persistent CTAs), profiles/pdl_mode3_ab_r02.log;
//   larger batches (cfg 3): off (+1.7 % padded but -7.6 % packed).
static thread_local int g_pdl_scope = 0;   // 0 = none, else the mode (1 / 3) of the innermost scope
struct PdlScope {
  const int prev;
  explicit PdlScope(int mode = 1) : prev(g_pdl_scope) { if (mode) g_pdl_scope = mode; }
  ~PdlScope() { g_pdl_scope = prev; }
};
int pdl_scope_exchange(int mode) {  // for the other translation units (train.cu): sets the mode, returns the previous one
  const int prev = g_pdl_scope;
  g_pdl_scope = mode;
  return prev;
}
// Sequence path: a step is ~90 kernels with a fixed cost of ~7 us each (B = 1: 685 us per step).  When the grids are a handful of
// CTAs the successor's prologue (barrier init, TMEM allocation, descriptor prefetch) can run on idle SMs under the predecessor:
// measured on B200 (profiles/pdl_small_r02.log) B = 1: 685 -> 616 us, B = 4: 711 -> 665 us per step; from B = 16 on the persistent
// kernels fill every SM and the early launch only costs (846 -> 919 us).  Hence: on up to 2048 stacked token rows.
static int pdl_auto_mode(long long rows) { return rows <= 2048 ? 1 : (rows <= 32768 ? 3 : 0); }
int pdl_mode() { return g_pdl_scope; }

// ---- debug-build guard bands (see common.cuh) -------------------------------------------------------------------------------
#ifdef SEQDIFF_DEBUG_BOUNDS
namespace {
struct GuardRec { const void* owner; void* p; };
std::vector<GuardRec> g_guards;
std::mutex g_guard_mu;
constexpr uint32_t kGuardWord = 0xA5C3F00Du;
__global__ void guard_fill_kernel(uint32_t* p) { p[threadIdx.x] = kGuardWord; }
__global__ void guard_check_kernel(uint32_t* const* bands, int n, int* broken) {
  const int i = blockIdx.x;
  if (i < n && bands[i][threadIdx.x] != kGuardWord) atomicAdd(broken, 1);
}
}  // namespace
int debug_guard_begin(const void* owner) {
  std::lock_guard<std::mutex> g(g_guard_mu);
  size_t w = 0;
  for (size_t i = 0; i < g_guards.size(); ++i)
    if (g_guards[i].owner != owner) g_guards[w++] = g_guards[i];
  g_guards.resize(w);
  return SEQDIFF_OK;
}
int debug_guard_add(const void* owner, void* p, cudaStream_t s) {
  {
    std::lock_guard<std::mutex> g(g_guard_mu);
    g_guards.push_back({owner, p});
  }
  guard_fill_kernel<<<1, 64, 0, s>>>(static_cast<uint32_t*>(p));  // capturable: re-armed by every replay of a captured step
  SD_CUDA(cudaGetLastError());
  return SEQDIFF_OK;
}
int debug_guard_check(cudaStream_t s, int* n_bands, int* n_broken) {
  std::vector<uint32_t*> h;
  {
    std::lock_guard<std::mutex> g(g_guard_mu);
    for (auto& r : g_guards) h.push_back(static_cast<uint32_t*>(r.p));
  }
  *n_bands = static_cast<int>(h.size());
  *n_broken = 0;
  if (h.empty()) return SEQDIFF_OK;
  SD_CUDA(cudaDeviceSynchronize());  // every stream: the bands belong to workspaces used on private streams as well
  if (const char* e = getenv("SEQDIFF_DEBUG_BREAK_GUARD"); e && e[0] == '1') SD_CUDA(cudaMemset(h[h.size() / 2], 0, 4));  // negative control of the check itself
  uint32_t** d = nullptr;
  int* cnt = nullptr;
  SD_CUDA(cudaMalloc(reinterpret_cast<void**>(&d), h.size() * sizeof(uint32_t*)));
  SD_CUDA(cudaMalloc(reinterpret_cast<void**>(&cnt), sizeof(int)));
  SD_CUDA(cudaMemcpy(d, h.data(), h.size() * sizeof(uint32_t*), cudaMemcpyHostToDevice));
  SD_CUDA(cudaMemset(cnt, 0, sizeof(int)));
  guard_check_kernel<<<static_cast<unsigned>(h.size()), 64, 0, s>>>(d, static_cast<int>(h.size()), cnt);
  SD_CUDA(cudaGetLastError());
  SD_CUDA(cudaStreamSynchronize(s));
  SD_CUDA(cudaMemcpy(n_broken, cnt, sizeof(int), cudaMemcpyDeviceToHost));
  cudaFree(d);
  cudaFree(cnt);
  return SEQDIFF_OK;
}
#else
int debug_guard_begin(const void*) { return SEQDIFF_OK; }
int debug_guard_add(const void*, void*, cudaStream_t) { return SEQDIFF_OK; }
int debug_guard_check(cudaStream_t, int* n_bands, int* n_broken) { *n_bands = 0; *n_broken = 0; return SEQDIFF_OK; }
#endif

int num_sms() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0)
      n = 148;
  }
  return n;
}

template <typename T> struct Fmt;  // operand format code of the tcgen05 instruction descriptor
template <> struct Fmt<f16> { static constexpr int v = 0; };
template <> struct Fmt<bf16> { static constexpr int v = 1; };
template <> struct Fmt<float> { static constexpr int v = -1; };  // fp32 mode: no 16-bit operand copies

template <typename T> static const T* pick(const Wt& w);
template <> const float* pick<float>(const Wt& w) { return w.f; }
template <> const bf16* pick<bf16>(const Wt& w) { return w.h; }
template <> const f16* pick<f16>(const Wt& w) { return w.g; }

// GEMM writing an operand-typed tensor (input of the next GEMM / attention); wfmt: weight format (0 fp16, 1 bf16)
static int gemm_T(int, int M, int N, int K, const float* A, const Wt& W, const float* bias, int epi, float* C, cudaStream_t s) {
  return gemm_f32(M, N, K, A, W.f, bias, nullptr, epi, C, s);
}
template <typename T>
static int gemm_T(int wfmt, int M, int N, int K, const T* A, const Wt& W, const float* bias, int epi, T* C, cudaStream_t s) {
  const void* w = wfmt == 1 ? static_cast<const void*>(W.h) : static_cast<const void*>(W.g);
  return gemm_16(M, N, K, A, Fmt<T>::v, w, wfmt, bias, nullptr, epi, C, Fmt<T>::v, s);
}
// GEMM writing the fp32 residual stream (LayerNorm input), optionally folding in the fp32 residual
static int gemm_S(int, int M, int N, int K, const float* A, const Wt& W, const float* bias, const float* resid, float* C, cudaStream_t s) {
  return gemm_f32(M, N, K, A, W.f, bias, resid, 0, C, s);
}
template <typename T>
static int gemm_S(int wfmt, int M, int N, int K, const T* A, const Wt& W, const float* bias, const float* resid, float* C, cudaStream_t s,
                  const LnResid* ln = nullptr) {
  const void* w = wfmt == 1 ? static_cast<const void*>(W.h) : static_cast<const void*>(W.g);
  return gemm_16(M, N, K, A, Fmt<T>::v, w, wfmt, bias, resid, 0, C, 2, s, 0, ln);
}
// Linear + residual (o, the fp32 stream) followed by its LayerNorm (h, the operand of the next GEMM; stats for a later LnResid rebuild).
// Fusing the LayerNorm into the GEMM epilogue was measured 2 % slower end to end at cfg 2 (DESIGN.md section 5c).
template <typename T>
static int gemm_ln(int wfmt, int M, int H, int K, const T* A, const Wt& W, const float* bias, const float* resid, float* o, const LnResid* lr,
                   const float* ln_w, const float* ln_b, float eps, T* h, float2* stats, cudaStream_t s) {
  SD_TRY(gemm_S(wfmt, M, H, K, A, W, bias, resid, o, s, lr));
  return layernorm<T>(o, M, H, ln_w, ln_b, eps, nullptr, h, stats, s);
}

__global__ void set_int_kernel(int* p, int v) {
  pdl_trigger();
  pdl_wait();
  *p = v;
}
// arms one sampling: step counter, arrival counter and the Philox key (seed, first global graph id) -- all read from device memory
// by the captured step graph, so the graph does not depend on them
__global__ void arm_loop_kernel(int* step, int v, uint64_t* rng, uint64_t seed, uint64_t gid0) {
  pdl_trigger();
  pdl_wait();
  step[0] = v;
  step[1] = 0;
  rng[0] = seed;
  rng[1] = gid0;
}

// =====================================================================================================
Model::~Model() {
  if (graph_exec) cudaGraphExecDestroy(graph_exec);
  if (score_exec) cudaGraphExecDestroy(score_exec);
  if (loop_stream) cudaStreamDestroy(loop_stream);
  if (ev_in) cudaEventDestroy(ev_in);
  if (ev_out) cudaEventDestroy(ev_out);
  for (void* p : allocs) cudaFree(p);
  for (void* p : packed_allocs) cudaFree(p);
  if (ws) { debug_guard_begin(ws); cudaFree(ws); }
  if (samp_in) { debug_guard_begin(samp_in); cudaFree(samp_in); }
  if (samp_inv) { debug_guard_begin(samp_inv); cudaFree(samp_inv); }
  if (score_in) { debug_guard_begin(score_in); cudaFree(score_in); }
  if (d_tables) cudaFree(d_tables);
  if (d_pack) cudaFree(d_pack);
  if (tws) { debug_guard_begin(tws); cudaFree(tws); }
  if (d_rp_tables) cudaFree(d_rp_tables);
}

void* Model::dalloc(size_t bytes) {
  if (packing && repack_reuse) {  // re-finalize after an optimizer step: same tensors, same order, same sizes -> same buffers
    if (packed_cursor < packed_allocs.size()) return packed_allocs[packed_cursor++];
    return nullptr;
  }
  void* p = nullptr;
  if (cudaMalloc(&p, bytes < 256 ? 256 : bytes) != cudaSuccess) return nullptr;
  (packing ? packed_allocs : allocs).push_back(p);
  return p;
}

static void add_schema(std::map<std::string, RawTensor>& raw, const std::string& name, int64_t numel) {
  RawTensor t;
  t.numel = numel;
  raw[name] = t;
}

int Model::init(const seqdiff_config_t& c, int dev, int arch_) {
  cfg = c;
  device = dev;
  arch = arch_;
  SD_CHECK(c.hidden_size % 256 == 0 && c.hidden_size >= 256 && c.hidden_size <= 1024, "hidden_size must be 256/512/768/1024");
  SD_CHECK(c.num_attention_heads * 64 == c.hidden_size, "head_dim must be 64");
  SD_CHECK(c.intermediate_size % 128 == 0, "intermediate_size must be a multiple of 128");
  SD_CHECK(c.num_hidden_layers >= 1 && c.max_position_embeddings >= 1, "bad layer count / max positions");
  SD_CHECK(c.feature_size >= 1 && c.feature_size <= 32, "feature_size must be in [1,32]");
  SD_CUDA(cudaSetDevice(dev));
  const int64_t H = c.hidden_size, I = c.intermediate_size, P = c.max_position_embeddings;
  // state_dict schema of ConditionalBertForDiffusionBase (SURVEY.md Appendix B)
  add_schema(raw, "timestep_projector.W", H / 2);
  auto emb_schema = [&](const std::string& p, int fin) {
    add_schema(raw, p + ".linear.weight", H * fin);
    add_schema(raw, p + ".linear.bias", H);
    add_schema(raw, p + ".LayerNorm.weight", H);
    add_schema(raw, p + ".LayerNorm.bias", H);
  };
  if (arch == kArchSequence)
    for (const char* side : {"ligand", "receptor"})
      for (auto kv : {std::pair<const char*, int>{"seq", 20}, std::pair<const char*, int>{"angle", 8}})
        emb_schema(std::string(side) + "_" + kv.first + "_embedding", kv.second);
  auto attn = [&](const std::string& p, bool rel) {
    for (const char* n : {"query", "key", "value"}) {
      add_schema(raw, p + ".self." + n + ".weight", H * H);
      add_schema(raw, p + ".self." + n + ".bias", H);
    }
    if (rel && c.relative_key) add_schema(raw, p + ".self.distance_embedding.weight", (2 * P - 1) * 64);
    add_schema(raw, p + ".output.dense.weight", H * H);
    add_schema(raw, p + ".output.dense.bias", H);
    add_schema(raw, p + ".output.LayerNorm.weight", H);
    add_schema(raw, p + ".output.LayerNorm.bias", H);
  };
  auto ffn_schema = [&](const std::string& p) {
    add_schema(raw, p + ".intermediate.dense.weight", I * H);
    add_schema(raw, p + ".intermediate.dense.bias", I);
    add_schema(raw, p + ".output.dense.weight", H * I);
    add_schema(raw, p + ".output.dense.bias", H);
    add_schema(raw, p + ".output.LayerNorm.weight", H);
    add_schema(raw, p + ".output.LayerNorm.bias", H);
  };
  const std::vector<const char*> se_blocks = arch == kArchSequence
                                                 ? std::vector<const char*>{"ligand_feature_emb", "receptor_feature_emb", "decoder_normalize"}
                                                 : std::vector<const char*>{"receptor_emb", "timestep_emb"};
  for (const char* blk : se_blocks) {
    const std::string p = blk;
    add_schema(raw, p + ".adaLN_modulation.0.weight", H * H);
    add_schema(raw, p + ".adaLN_modulation.0.bias", H);
    add_schema(raw, p + ".adaLN_modulation.2.weight", 6 * H * H);
    add_schema(raw, p + ".adaLN_modulation.2.bias", 6 * H);
    attn(p + ".attn", true);
    add_schema(raw, p + ".mlp.0.weight", 4 * H * H);
    add_schema(raw, p + ".mlp.0.bias", 4 * H);
    add_schema(raw, p + ".mlp.3.weight", 4 * H * H);
    add_schema(raw, p + ".mlp.3.bias", H);
  }
  for (int i = 0; i < c.num_hidden_layers; ++i) {
    const std::string p = "decoder.layer." + std::to_string(i);
    attn(p + ".attention", true);
    attn(p + ".crossattention", false);
    ffn_schema(p);
  }
  if (arch == kArchStructure) {  // structure_model/model.py:163-178
    emb_schema("receptor_seq_emb", 20);
    emb_schema("receptor_angle_emb", c.feature_size);
    emb_schema("ligand_angle_emb", c.feature_size);
    for (int i = 0; i < c.num_hidden_layers; ++i) {
      const std::string p = "encoder.layer." + std::to_string(i);
      attn(p + ".attention", true);
      ffn_schema(p);
    }
  }
  const std::string head = arch == kArchSequence ? "amino_acid_predictor" : "angles_predictor";
  add_schema(raw, head + ".dense1.weight", H * H);
  add_schema(raw, head + ".dense1.bias", H);
  add_schema(raw, head + ".layer_norm.weight", H);
  add_schema(raw, head + ".layer_norm.bias", H);
  add_schema(raw, head + ".dense2.weight", static_cast<int64_t>(c.feature_size) * H);
  add_schema(raw, head + ".dense2.bias", c.feature_size);
  d_step = static_cast<int*>(dalloc(256));  // [0] step counter of the sampling loop, [1] arrival counter of its reverse step
  SD_CHECK(d_step != nullptr, "cudaMalloc failed");
  SD_CUDA(cudaMemset(d_step, 0, 256));
  return SEQDIFF_OK;
}

int Model::set_tensor(const char* name, const float* data, int64_t numel, cudaStream_t s) {
  auto it = raw.find(name);
  if (it == raw.end()) {
    set_error(std::string("unknown tensor name: ") + name);
    return SEQDIFF_ERR_STATE;
  }
  RawTensor& t = it->second;
  if (t.numel != numel) {
    set_error(std::string("size mismatch for ") + name + ": expected " + std::to_string(t.numel) + ", got " + std::to_string(numel));
    return SEQDIFF_ERR_INVALID;
  }
  // receptor_feature_emb is dead weight in the reference (quirk Q1): accepted, never stored.
  if (arch == kArchSequence && std::strncmp(name, "receptor_feature_emb.", 21) == 0) {
    t.set = true;
    return SEQDIFF_OK;
  }
  if (!t.ptr) {
    t.ptr = static_cast<float*>(dalloc(static_cast<size_t>(numel) * sizeof(float)));
    SD_CHECK(t.ptr != nullptr, "cudaMalloc failed");
  }
  SD_CUDA(cudaMemcpyAsync(t.ptr, data, static_cast<size_t>(numel) * sizeof(float), cudaMemcpyDefault, s));
  t.set = true;
  finalized = false;
  return SEQDIFF_OK;
}

// ---- batched refresh of the packed weight copies after an optimizer step ---------------------------------------------------------
namespace {
struct RpChunk { const float* src; void* a; void* b; int n, rows, cols, r0; };  // copy / convert: n elements; transpose: a 64 x 64 tile at (r0, cols-offset in n)
__global__ void __launch_bounds__(256) rp_copy_kernel(const RpChunk* __restrict__ tab) {
  const RpChunk c = tab[blockIdx.x];
  float* dst = static_cast<float*>(c.a);
  for (int i = threadIdx.x * 4; i < c.n; i += 1024) {
    if (i + 3 < c.n) *reinterpret_cast<float4*>(dst + i) = *reinterpret_cast<const float4*>(c.src + i);
    else for (int j = i; j < c.n; ++j) dst[j] = c.src[j];
  }
}
__global__ void __launch_bounds__(256) rp_conv_kernel(const RpChunk* __restrict__ tab) {  // fp32 -> bf16 (a) and fp16 (b), n % 4 == 0 per chunk start
  const RpChunk c = tab[blockIdx.x];
  bf16* h = static_cast<bf16*>(c.a);
  f16* g = static_cast<f16*>(c.b);
  for (int i = threadIdx.x * 4; i < c.n; i += 1024) {
    if (i + 3 < c.n) {
      const float4 v = *reinterpret_cast<const float4*>(c.src + i);
      *reinterpret_cast<uint2*>(h + i) = make_uint2(pack_bf16x2(v.x, v.y), pack_bf16x2(v.z, v.w));
      *reinterpret_cast<uint2*>(g + i) = make_uint2(pack_f16x2(v.x, v.y), pack_f16x2(v.z, v.w));
    } else {
      for (int j = i; j < c.n; ++j) { h[j] = from_f32<bf16>(c.src[j]); g[j] = from_f32<f16>(c.src[j]); }
    }
  }
}
template <typename T>
__global__ void __launch_bounds__(256) rp_trans_kernel(const RpChunk* __restrict__ tab) {  // fp32 [rows, cols] -> T [cols, rows], one 64 x 64 tile per block
  __shared__ float tile[64][65];
  const RpChunk c = tab[blockIdx.x];
  T* out = static_cast<T*>(c.a);
  const int r0 = c.r0, c0 = c.n;
  const int tx = threadIdx.x & 63, ty = threadIdx.x >> 6;
#pragma unroll 4
  for (int i = ty; i < 64; i += 4) {
    const int r = r0 + i, cc = c0 + tx;
    tile[i][tx] = (r < c.rows && cc < c.cols) ? c.src[static_cast<size_t>(r) * c.cols + cc] : 0.f;
  }
  __syncthreads();
#pragma unroll 4
  for (int i = ty; i < 64; i += 4) {
    const int cc = c0 + i, r = r0 + tx;
    if (cc < c.cols && r < c.rows) out[static_cast<size_t>(cc) * c.rows + r] = from_f32<T>(tile[tx][i]);
  }
}
}  // namespace

int Model::repack_fast(cudaStream_t s) {
  constexpr int kChunk = 8192;
  if (!d_rp_tables || rp_table_prec != train_prec) {
    std::vector<RpChunk> tab;
    for (const RpCopy& o : rp_copy)
      for (int64_t off = 0; off < o.n; off += kChunk)
        tab.push_back({o.src + off, o.dst + off, nullptr, static_cast<int>(o.n - off < kChunk ? o.n - off : kChunk), 0, 0, 0});
    rp_n_copy = static_cast<int>(tab.size());
    for (const RpConv& o : rp_conv)
      for (int64_t off = 0; off < o.n; off += kChunk)
        tab.push_back({o.src + off, static_cast<bf16*>(o.h) + off, static_cast<f16*>(o.g) + off, static_cast<int>(o.n - off < kChunk ? o.n - off : kChunk), 0, 0, 0});
    rp_n_conv = static_cast<int>(tab.size()) - rp_n_copy;
    auto tiles = [&](const std::vector<RpTrans>& ops) {
      for (const RpTrans& o : ops)
        for (int r0 = 0; r0 < o.rows; r0 += 64)
          for (int c0 = 0; c0 < o.cols; c0 += 64) tab.push_back({o.src, o.dst, nullptr, c0, o.rows, o.cols, r0});
    };
    const size_t before = tab.size();
    tiles(rp_trans);
    rp_n_trans = static_cast<int>(tab.size() - before);
    tiles(rp_trans_f32);
    rp_n_trans_f32 = static_cast<int>(tab.size() - before) - rp_n_trans;
    if (d_rp_tables) { SD_CUDA(cudaDeviceSynchronize()); SD_CUDA(cudaFree(d_rp_tables)); d_rp_tables = nullptr; }
    SD_CUDA(cudaMalloc(&d_rp_tables, tab.size() * sizeof(RpChunk)));
    SD_CUDA(cudaMemcpyAsync(d_rp_tables, tab.data(), tab.size() * sizeof(RpChunk), cudaMemcpyHostToDevice, s));
    SD_CUDA(cudaStreamSynchronize(s));  // tab is a stack-lifetime host buffer
    rp_table_prec = train_prec;
  }
  const RpChunk* t = static_cast<const RpChunk*>(d_rp_tables);
  if (rp_n_copy) { SD_CUDA(launch_k(rp_copy_kernel, dim3(rp_n_copy), dim3(256), 0, s, t)); SD_LAUNCHED("repack_copy", s); }
  t += rp_n_copy;
  if (rp_n_conv) { SD_CUDA(launch_k(rp_conv_kernel, dim3(rp_n_conv), dim3(256), 0, s, t)); SD_LAUNCHED("repack_convert", s); }
  t += rp_n_conv;
  if (rp_n_trans) {
    if (train_prec == SEQDIFF_FP32) SD_CUDA(launch_k(rp_trans_kernel<float>, dim3(rp_n_trans), dim3(256), 0, s, t));
    else if (train_prec == SEQDIFF_BF16) SD_CUDA(launch_k(rp_trans_kernel<bf16>, dim3(rp_n_trans), dim3(256), 0, s, t));
    else SD_CUDA(launch_k(rp_trans_kernel<f16>, dim3(rp_n_trans), dim3(256), 0, s, t));
    SD_LAUNCHED("repack_transpose", s);
  }
  t += rp_n_trans;
  if (rp_n_trans_f32) { SD_CUDA(launch_k(rp_trans_kernel<float>, dim3(rp_n_trans_f32), dim3(256), 0, s, t)); SD_LAUNCHED("repack_transpose", s); }
  return SEQDIFF_OK;
}

int Model::finalize(cudaStream_t s) {
  for (auto& kv : raw)
    if (!kv.second.set) {
      set_error("tensor never set: " + kv.first);
      return SEQDIFF_ERR_STATE;
    }
  if (!repack_reuse) {
    if (graph_exec) {  // the packed copies are re-allocated: a captured graph would hold stale pointers
      cudaGraphExecDestroy(graph_exec);
      graph_exec = nullptr;
      graph_key = GraphKey();
    }
    if (score_exec) {
      cudaGraphExecDestroy(score_exec);
      score_exec = nullptr;
      score_key = GraphKey();
    }
    if (!packed_allocs.empty()) {  // re-finalize after a weight upload: drop the previous packed copies
      SD_CUDA(cudaDeviceSynchronize());
      for (void* p : packed_allocs) cudaFree(p);
      packed_allocs.clear();
    }
  }
  if (repack_reuse && !rp_conv.empty()) return repack_fast(s);  // same buffers, same operations: the batched refresh
  packed_cursor = 0;
  packing = true;
  rp_copy.clear(); rp_conv.clear(); rp_trans.clear(); rp_trans_f32.clear();
  rp_table_prec = -2;
  const int64_t H = cfg.hidden_size, I = cfg.intermediate_size, P = cfg.max_position_embeddings;
  int rc = SEQDIFF_OK;
  auto R = [&](const std::string& n) -> const float* { return raw.at(n).ptr; };
  // fp32 matrix -> Wt with bf16 and fp16 copies
  // training: every GEMM weight also gets its transposed copy in the operand type of the training precision
  auto transposed = [&](Wt& w, int64_t rows, int64_t cols) {
    w.rows = rows;
    w.cols = cols;
    if (train_prec < 0) return;
    const size_t n = static_cast<size_t>(rows) * cols;
    void* t = dalloc(n * (train_prec == SEQDIFF_FP32 ? 4 : 2));
    int r = SEQDIFF_ERR_CUDA;
    if (t) {
      if (train_prec == SEQDIFF_FP32) r = transpose_cast<float>(w.f, static_cast<int>(rows), static_cast<int>(cols), static_cast<float*>(t), s);
      else if (train_prec == SEQDIFF_BF16) r = transpose_cast<bf16>(w.f, static_cast<int>(rows), static_cast<int>(cols), static_cast<bf16*>(t), s);
      else r = transpose_cast<f16>(w.f, static_cast<int>(rows), static_cast<int>(cols), static_cast<f16*>(t), s);
    }
    if (r != SEQDIFF_OK) rc = SEQDIFF_ERR_CUDA;
    w.t = t;
    rp_trans.push_back({w.f, t, static_cast<int>(rows), static_cast<int>(cols)});
  };
  auto both = [&](const float* f, int64_t n) -> Wt {
    Wt w;
    w.f = f;
    bf16* h = static_cast<bf16*>(dalloc(static_cast<size_t>(n) * sizeof(bf16)));
    f16* g = static_cast<f16*>(dalloc(static_cast<size_t>(n) * sizeof(f16)));
    if (!h || !g || f32_to_16<bf16>(f, static_cast<size_t>(n), h, s) != SEQDIFF_OK ||
        f32_to_16<f16>(f, static_cast<size_t>(n), g, s) != SEQDIFF_OK)
      rc = SEQDIFF_ERR_CUDA;
    w.h = h;
    w.g = g;
    rp_conv.push_back({f, h, g, n});
    return w;
  };
  // stack several [rows_i, cols] fp32 tensors (row-wise) into a fresh buffer
  auto stack = [&](const std::vector<const float*>& parts, int64_t each) -> float* {
    float* dst = static_cast<float*>(dalloc(parts.size() * static_cast<size_t>(each) * sizeof(float)));
    if (!dst) { rc = SEQDIFF_ERR_CUDA; return nullptr; }
    for (size_t i = 0; i < parts.size(); ++i) {
      if (cudaMemcpyAsync(dst + i * each, parts[i], static_cast<size_t>(each) * sizeof(float), cudaMemcpyDeviceToDevice, s) != cudaSuccess)
        rc = SEQDIFF_ERR_CUDA;
      rp_copy.push_back({dst + i * each, parts[i], each});
    }
    return dst;
  };
  auto emb = [&](const std::string& p, int fin) -> EmbW {
    EmbW e;
    e.fin = fin;
    float* wt = static_cast<float*>(dalloc(static_cast<size_t>(H) * fin * sizeof(float)));
    if (!wt || transpose_f32(R(p + ".linear.weight"), static_cast<int>(H), fin, wt, s) != SEQDIFF_OK) rc = SEQDIFF_ERR_CUDA;
    e.Wt_ = wt;
    rp_trans_f32.push_back({R(p + ".linear.weight"), wt, static_cast<int>(H), fin});
    e.b = R(p + ".linear.bias");
    e.ln_w = R(p + ".LayerNorm.weight");
    e.ln_b = R(p + ".LayerNorm.bias");
    return e;
  };
  auto attn = [&](const std::string& p, bool self_rel) -> AttnW {
    AttnW a;
    const float* w = stack({R(p + ".self.query.weight"), R(p + ".self.key.weight"), R(p + ".self.value.weight")}, H * H);
    a.qkv = both(w, 3 * H * H);
    transposed(a.qkv, 3 * H, H);
    a.qkv_b = stack({R(p + ".self.query.bias"), R(p + ".self.key.bias"), R(p + ".self.value.bias")}, H);
    if (self_rel && cfg.relative_key) a.E = both(R(p + ".self.distance_embedding.weight"), (2 * P - 1) * 64);
    a.out = both(R(p + ".output.dense.weight"), H * H);
    transposed(a.out, H, H);
    a.out_b = R(p + ".output.dense.bias");
    a.ln_w = R(p + ".output.LayerNorm.weight");
    a.ln_b = R(p + ".output.LayerNorm.bias");
    return a;
  };
  auto se = [&](const std::string& p) -> SEW {
    SEW w;
    w.ada0 = both(R(p + ".adaLN_modulation.0.weight"), H * H);
    transposed(w.ada0, H, H);
    w.ada0_b = R(p + ".adaLN_modulation.0.bias");
    w.ada2 = both(R(p + ".adaLN_modulation.2.weight"), 6 * H * H);
    transposed(w.ada2, 6 * H, H);
    w.ada2_b = R(p + ".adaLN_modulation.2.bias");
    w.attn = attn(p + ".attn", true);
    w.m0 = both(R(p + ".mlp.0.weight"), 4 * H * H);
    transposed(w.m0, 4 * H, H);
    w.m0_b = R(p + ".mlp.0.bias");
    w.m3 = both(R(p + ".mlp.3.weight"), 4 * H * H);
    transposed(w.m3, H, 4 * H);
    w.m3_b = R(p + ".mlp.3.bias");
    return w;
  };
  ts_W = R("timestep_projector.W");
  auto ffn = [&](const std::string& p, LayerW& l) {
    l.inter = both(R(p + ".intermediate.dense.weight"), I * H);
    transposed(l.inter, I, H);
    l.inter_b = R(p + ".intermediate.dense.bias");
    l.outd = both(R(p + ".output.dense.weight"), H * I);
    transposed(l.outd, H, I);
    l.outd_b = R(p + ".output.dense.bias");
    l.oln_w = R(p + ".output.LayerNorm.weight");
    l.oln_b = R(p + ".output.LayerNorm.bias");
  };
  enc_layers.clear();
  if (arch == kArchSequence) {
    lig_seq = emb("ligand_seq_embedding", 20);
    lig_ang = emb("ligand_angle_embedding", 8);
    rec_seq = emb("receptor_seq_embedding", 20);
    rec_ang = emb("receptor_angle_embedding", 8);
    se_lig = se("ligand_feature_emb");
    se_dec = se("decoder_normalize");
  } else {  // structure model: se_lig = receptor_emb (x = angles, c = sequence), se_dec = timestep_emb
    rec_seq = emb("receptor_seq_emb", 20);
    rec_ang = emb("receptor_angle_emb", cfg.feature_size);
    lig_ang = emb("ligand_angle_emb", cfg.feature_size);
    se_lig = se("receptor_emb");
    se_dec = se("timestep_emb");
    for (int i = 0; i < cfg.num_hidden_layers; ++i) {
      const std::string p = "encoder.layer." + std::to_string(i);
      LayerW l;
      l.self = attn(p + ".attention", true);
      ffn(p, l);
      enc_layers.push_back(l);
    }
  }
  layers.clear();
  std::vector<const float*> ckv_w, ckv_b;
  for (int i = 0; i < cfg.num_hidden_layers; ++i) {
    const std::string p = "decoder.layer." + std::to_string(i);
    LayerW l;
    l.self = attn(p + ".attention", true);
    l.cq = both(R(p + ".crossattention.self.query.weight"), H * H);
    transposed(l.cq, H, H);
    l.cq_b = R(p + ".crossattention.self.query.bias");
    ckv_w.push_back(R(p + ".crossattention.self.key.weight"));
    ckv_w.push_back(R(p + ".crossattention.self.value.weight"));
    ckv_b.push_back(R(p + ".crossattention.self.key.bias"));
    ckv_b.push_back(R(p + ".crossattention.self.value.bias"));
    l.cout = both(R(p + ".crossattention.output.dense.weight"), H * H);
    transposed(l.cout, H, H);
    l.cout_b = R(p + ".crossattention.output.dense.bias");
    l.cln_w = R(p + ".crossattention.output.LayerNorm.weight");
    l.cln_b = R(p + ".crossattention.output.LayerNorm.bias");
    ffn(p, l);
    layers.push_back(l);
  }
  ckv_all = both(stack(ckv_w, H * H), static_cast<int64_t>(ckv_w.size()) * H * H);
  transposed(ckv_all, static_cast<int64_t>(ckv_w.size()) * H, H);
  ckv_all_b = stack(ckv_b, H);
  const std::string head = arch == kArchSequence ? "amino_acid_predictor" : "angles_predictor";
  p1 = both(R(head + ".dense1.weight"), H * H);
  transposed(p1, H, H);
  p1_b = R(head + ".dense1.bias");
  p_ln_w = R(head + ".layer_norm.weight");
  p_ln_b = R(head + ".layer_norm.bias");
  p2_w = R(head + ".dense2.weight");
  p2_b = R(head + ".dense2.bias");
  packing = false;
  if (rc != SEQDIFF_OK) {
    set_error("finalize: allocation or packing kernel failed");
    return rc;
  }
  finalized = true;
  return SEQDIFF_OK;
}

// =====================================================================================================
// workspace
// =====================================================================================================
static size_t align256(size_t b) { return (b + 255) & ~static_cast<size_t>(255); }

size_t Model::workspace_need(int precision, int B, int Ll, int Lr) const {
  const size_t es = precision == SEQDIFF_FP32 ? 4 : 2;       // operand element size
  const size_t dual = precision == SEQDIFF_FP32 ? 4 : 4 + 2;  // fp32 stream (+ 16-bit operand copy)
  const size_t H = cfg.hidden_size, I = cfg.intermediate_size, NL = cfg.num_hidden_layers;
  const size_t Ml = static_cast<size_t>(B) * Ll, Mr = static_cast<size_t>(B) * Lr, Mt = Ml + Mr;
  size_t n = 0;
  n += 2 * align256(static_cast<size_t>(B) * H * 4);  // te fp32 + operand copy
  n += align256((Ml + Mr) * 4);                       // stacked masks
  n += 3 * (align256(Mt * H * 4) + align256(Mt * H * 2));  // x, x1, x2 (stream + operand)
  n += 2 * align256(Mt * H * 4);                      // o, m2 (fp32, LayerNorm inputs)
  n += 3 * align256(Mt * H * es);                     // c, u, ctx
  n += align256(Mt * 6 * H * es);                     // mod
  n += align256(Mt * 3 * H * es);                     // qkv
  n += align256(Mt * 4 * H * es);                     // m1
  n += align256(Mr * NL * 2 * H * es);                // kv_all
  n += 2 * (align256(Ml * H * 4) + align256(Ml * H * 2));  // decoder h ping-pong
  n += 2 * align256(Ml * H * es);                     // cq, y
  n += align256(Ml * H * 4) + align256(Ml * 3 * 8);   // third pre-LN buffer, LayerNorm row statistics
  n += align256(Ml * I * es);                         // ffn
  (void)dual;
  return n + 8192 + 64 * kGuardBytes;  // (debug build: one guard band per carved buffer)
}

int Model::ensure_workspace(size_t bytes) {
  if (bytes <= ws_bytes) return SEQDIFF_OK;
  if (ws) {
    SD_CUDA(cudaDeviceSynchronize());
    debug_guard_begin(ws);  // (debug build) the bands of the old workspace go with it
    SD_CUDA(cudaFree(ws));
    ws = nullptr;
    ws_bytes = 0;
  }
  SD_CUDA(cudaMalloc(reinterpret_cast<void**>(&ws), bytes));
  ws_bytes = bytes;
  return SEQDIFF_OK;
}

struct Bump {
  uint8_t* p;
  cudaStream_t gs;    // debug build: stream the guard bands are filled on
  const void* owner;  // debug build: the carve these bands belong to (a new carve of the same workspace replaces them)
  explicit Bump(uint8_t* base, cudaStream_t s = nullptr) : p(base), gs(s), owner(base) { debug_guard_begin(owner); }
  template <typename T> T* take(size_t n) {
    T* r = reinterpret_cast<T*>(p);
    p += align256(n * sizeof(T));
    if (kGuardBytes) {
      debug_guard_add(owner, p, gs);
      p += kGuardBytes;
    }
    return r;
  }
};

// a residual-stream tensor: fp32 master (s) + operand-typed copy (t) fed to the next GEMM.
// In fp32 mode both are the same buffer and the rowwise kernels write it once.
template <typename T> struct Act {
  float* s = nullptr;
  T* t = nullptr;
  T* t_out() const { return t; }
};
template <> struct Act<float> {
  float* s = nullptr;
  float* t = nullptr;
  float* t_out() const { return nullptr; }  // already written through `s`
};
template <typename T> static Act<T> take_act(Bump& bp, size_t n) {
  Act<T> a;
  a.s = bp.take<float>(n);
  a.t = bp.take<T>(n);
  return a;
}
template <> Act<float> take_act<float>(Bump& bp, size_t n) {
  Act<float> a;
  a.s = bp.take<float>(n);
  a.t = a.s;
  return a;
}
template <typename T> static Act<T> offset(const Act<T>& a, size_t n) {
  Act<T> r;
  r.s = a.s + n;
  r.t = a.t + n;
  return r;
}

// =====================================================================================================
// forward
// =====================================================================================================
template <typename T> struct SEBufs {
  T *u, *mod, *qkv, *ctx, *m1;
  float *o, *m2;
  Act<T> x1;
};

// Sampling loop: what se_layer takes from the per-sampling invariants (LoopInv).  o_hi != NULL: only rows [0, Ma) go through the
// attention sublayer (segs cover just those); rows r >= Ma take its output (dense + residual, before the LayerNorm) and their
// residual x from row r - Ma of o_hi / x_hi.  mod != NULL: the adaLN GEMMs are skipped and every row takes row *mod_row of mod.
template <typename T> struct SEHoist {
  int Ma;
  const float* o_hi;
  const float* x_hi;
  const T* mod;
  const int* mod_row;
};

// SELayer.forward (model.py:52-63).  x:[M,H]; c:[Mc,H] with token row r using c row r / mod_div.
// packs (optional, one per segment): ragged batch -- the segment's graphs are addressed through offset / length arrays (absolute rows
// of the token matrix) and seg.L is the largest length; row_graph: graph of every row (conditioning broadcast over a graph).
template <typename T>
static int se_layer(const Model& m, int wfmt, const SEW& w, const Act<T>& x, const T* c, int Mc, int mod_div, int M,
                    const std::vector<Segment>& segs, const SEBufs<T>& b, const Act<T>& out, cudaStream_t s,
                    const std::vector<AttnPack>* packs = nullptr, const int* row_graph = nullptr, const SEHoist<T>* hz = nullptr) {
  const int H = m.cfg.hidden_size, P = m.cfg.max_position_embeddings, heads = m.cfg.num_attention_heads;
  const int Ma = hz && hz->o_hi ? hz->Ma : M;
  const T* mod = hz && hz->mod ? hz->mod : b.mod;
  const int* mod_row = hz ? hz->mod_row : nullptr;
  if (mod == b.mod) {
    SD_TRY(gemm_T(wfmt, Mc, H, H, c, w.ada0, w.ada0_b, 2, b.u, s));          // SiLU(Linear(c))
    SD_TRY(gemm_T(wfmt, Mc, 6 * H, H, b.u, w.ada2, w.ada2_b, 0, b.mod, s));   // -> 6 chunks
  }
  SD_TRY(gemm_T(wfmt, Ma, 3 * H, H, x.t, w.attn.qkv, w.attn.qkv_b, 0, b.qkv, s));
  for (size_t gi = 0; gi < segs.size(); ++gi) {
    const Segment& g = segs[gi];
    const T* base = b.qkv + static_cast<size_t>(g.row0) * 3 * H;
    SD_TRY(attention<T>(g.B, heads, g.L, g.L, base, 3 * H, base + H, 3 * H, base + 2 * H, 3 * H, pick<T>(w.attn.E), P, g.mask,
                        b.ctx + static_cast<size_t>(g.row0) * H, s, packs ? &(*packs)[gi] : nullptr));
  }
  SD_TRY(gemm_S(wfmt, Ma, H, H, b.ctx, w.attn.out, w.attn.out_b, x.s, b.o, s));  // dense + residual (fp32)
  SD_TRY(ln_modulate<T>(b.o, M, H, true, w.attn.ln_w, w.attn.ln_b, m.cfg.layer_norm_eps, x.s, mod, mod_div, 0, b.x1.s, b.x1.t_out(), s, row_graph,
                        mod_row, Ma, hz ? hz->o_hi : nullptr, hz ? hz->x_hi : nullptr));
  SD_TRY(gemm_T(wfmt, M, 4 * H, H, b.x1.t, w.m0, w.m0_b, 1, b.m1, s));        // GELU
  SD_TRY(gemm_S(wfmt, M, H, 4 * H, b.m1, w.m3, w.m3_b, nullptr, b.m2, s));
  SD_TRY(ln_modulate<T>(b.m2, M, H, false, nullptr, nullptr, 0.f, b.x1.s, mod, mod_div, 3, out.s, out.t_out(), s, row_graph, mod_row));
  return SEQDIFF_OK;
}

// The forward's workspace carve.  loop_invariants_t takes its scratch from the same carve, so the debug build's guard bands stay
// the ones the replayed step writes around.
template <typename T> struct FwdBufs {
  float* te;
  T* teT;
  float* maskcat;
  Act<T> x;   // embeddings; reused as the decoder_normalize output
  Act<T> x2;  // ligand_feature_emb output: [lig | rec]
  SEBufs<T> sb;
  T *ccat, *kv_all;
  Act<T> hbuf[2];
  float* obuf3;     // third rotating pre-LN buffer (16-bit modes)
  float2* lnstats;  // (mean, rstd) of the three LayerNorms of a layer
  T *cq, *y, *ffn;
};
template <typename T>
static FwdBufs<T> carve_forward(uint8_t* ws, cudaStream_t s, int B, int H, int I, int NL, int Mlp, int Mrp, int Ml, int Mr) {
  constexpr bool k16 = !std::is_same<T, float>::value;
  const size_t MtH = static_cast<size_t>(Ml + Mr) * H, MlH = static_cast<size_t>(Ml) * H;
  Bump bp(ws, s);
  FwdBufs<T> f;
  f.te = bp.take<float>(static_cast<size_t>(B) * H);
  f.teT = k16 ? bp.take<T>(static_cast<size_t>(B) * H) : reinterpret_cast<T*>(f.te);
  f.maskcat = bp.take<float>(static_cast<size_t>(Mlp) + Mrp);
  f.x = take_act<T>(bp, MtH);
  f.x2 = take_act<T>(bp, MtH);
  f.sb.x1 = take_act<T>(bp, MtH);
  f.sb.o = bp.take<float>(MtH);
  f.sb.m2 = bp.take<float>(MtH);
  f.ccat = bp.take<T>(MtH);
  f.sb.u = bp.take<T>(MtH);
  f.sb.ctx = bp.take<T>(MtH);
  f.sb.mod = bp.take<T>(MtH * 6);
  f.sb.qkv = bp.take<T>(MtH * 3);
  f.sb.m1 = bp.take<T>(MtH * 4);
  f.kv_all = bp.take<T>(static_cast<size_t>(Mr) * NL * 2 * H);
  f.hbuf[0] = take_act<T>(bp, MlH);
  f.hbuf[1] = take_act<T>(bp, MlH);
  f.obuf3 = bp.take<float>(MlH);
  f.lnstats = bp.take<float2>(3 * static_cast<size_t>(Ml));
  f.cq = bp.take<T>(MlH);
  f.y = bp.take<T>(MlH);
  f.ffn = bp.take<T>(static_cast<size_t>(Ml) * I);
  return f;
}


template <typename T>
int Model::forward_t(int wfmt, int B, int Ll, int Lr, const float* timestep, const int* step_ptr, const float* x_t,
                     const float* lig_angle, const float* lig_mask, const float* rec_seq_in, const float* rec_angle,
                     const float* rec_mask, float* logits, cudaStream_t s, const PackInfo* pk, const LoopInv* inv, int K) {
  constexpr bool k16 = !std::is_same<T, float>::value;
  const int H = cfg.hidden_size, I = cfg.intermediate_size, NL = cfg.num_hidden_layers, heads = cfg.num_attention_heads;
  const int P = cfg.max_position_embeddings;
  const float eps = cfg.layer_norm_eps;
  // packed (ragged) batch: only the valid prefix of every graph is a row; inputs, masks and logits keep their padded layouts.
  // The receptor rows are those of the B / K pockets.  A receptor-only pack (pk->lig_padded, sampling loop) packs the receptor
  // rows alone: pl, the pack the ligand side uses, is then NULL and the ligand rows run the padded path.
  const PackInfo* pl = pk && !pk->lig_padded ? pk : nullptr;
  const int Ml = pk ? pk->Ml : B * Ll, Mr = pk ? pk->Mr : B / K * Lr, Mt = Ml + Mr;
  const int Mlp = B * Ll, Mrp = B / K * Lr;  // padded row counts (input tensors, key masks)
  const size_t MlH = static_cast<size_t>(Ml) * H;
  const FwdBufs<T> f = carve_forward<T>(ws, s, B, H, I, NL, Mlp, Mrp, Ml, Mr);
  float* te = f.te;
  T* teT = f.teT;
  const Act<T> x = f.x, x2 = f.x2;
  SEBufs<T> sb = f.sb;
  T *ccat = f.ccat, *kv_all = f.kv_all, *cq = f.cq, *y = f.y, *ffn = f.ffn;
  const Act<T>* hbuf = f.hbuf;
  float2* lnstats = f.lnstats;

  // timestep features + the four BertEmbeddings (model.py:211-213,219-220).  Sampling loop (inv): the receptor sequence embedding
  // and the timestep features of every step are in inv; the angle embeddings stay here, because c = LN(Linear(angles)) + te is
  // rounded to the operand type after the add.
  if (!inv) SD_TRY(timestep_embed(timestep, step_ptr, ts_W, B, H, te, k16 ? static_cast<void*>(teT) : nullptr, Fmt<T>::v, s));
  const Act<T> xr = offset(x, MlH);
  {
    const float* te_ = inv ? inv->te : te;
    auto job = [&](const float* in, int M, const EmbW& e, bool cond, int L, float* o32, T* oT, bool lig) {
      EmbedJob jb{};
      jb.x = in; jb.Wt = e.Wt_; jb.b = e.b; jb.lnw = e.ln_w; jb.lnb = e.ln_b; jb.te = cond ? te_ : nullptr;
      jb.te_row = cond && inv ? step_ptr : nullptr;
      jb.out32 = o32; jb.outT = oT; jb.M = M; jb.fin = e.fin; jb.L = L;
      if (lig ? pl : pk) {
        jb.src_rows = lig ? pk->src_l : pk->src_r;
        jb.row_graph = lig ? pk->graph : pk->graph + pk->Ml;
      }
      return jb;
    };
    EmbedJobs jobs{};
    jobs.j[jobs.n++] = job(x_t, Ml, lig_seq, false, Ll, x.s, x.t_out(), true);
    if (!inv) jobs.j[jobs.n++] = job(rec_seq_in, Mr, rec_seq, false, Lr, xr.s, xr.t_out(), false);
    // the conditioning c = LN(Linear(angles)) + te only ever feeds a GEMM: operand type only
    jobs.j[jobs.n++] = job(lig_angle, Ml, lig_ang, true, Ll, k16 ? nullptr : reinterpret_cast<float*>(ccat), k16 ? ccat : nullptr, true);
    jobs.j[jobs.n++] = job(rec_angle, Mr, rec_ang, true, Lr, k16 ? nullptr : reinterpret_cast<float*>(ccat + MlH), k16 ? ccat + MlH : nullptr, false);
    if (Ll == Lr && !inv) {  // stacked [lig | rec] key mask for the one-pass ligand_feature_emb attention (always the PADDED masks)
      jobs.cat_dst = f.maskcat; jobs.cat_a = lig_mask; jobs.cat_b = rec_mask; jobs.cat_na = Mlp; jobs.cat_nb = Mrp;
    }
    SD_TRY(embed_ln_multi<T>(jobs, eps, H, s));
  }

  // ligand_feature_emb on ligand AND receptor tokens in one pass (model.py:214-224, quirk Q1).  Sampling loop: its attention
  // sublayer sees the receptor embedding alone (the conditioning enters after it), so only the ligand rows run through it here and
  // the receptor rows of its output come from inv->o.
  std::vector<Segment> segs;
  std::vector<AttnPack> packs;
  AttnPack pk_self{}, pk_cross{};
  if (pk) {  // receptor-only pack: the cross-attention's queries are the padded ligand rows (off_l[b] = b * Ll, len_l[b] = Ll)
    pk_self = AttnPack{pk->off_l, pk->off_l, pk->len_l, Ml, Ml, Ll};
    pk_cross = AttnPack{pk->off_l, pk->off_r, pk->len_l, Ml, Mr, Lr};
  }
  SD_CHECK(pl == pk || inv, "a receptor-only pack exists in the sampling loop only");
  if (inv) {
    segs.push_back({0, B, pl ? pl->max_l : Ll, lig_mask});
    if (pl) packs.push_back(pk_self);
  } else if (pk) {
    // offsets are absolute rows of the stacked matrix, so every segment starts at row 0
    if (Ll == Lr) {
      segs.push_back({0, 2 * B, pk->max_l > pk->max_r ? pk->max_l : pk->max_r, f.maskcat});
      packs.push_back(AttnPack{pk->off_cat, pk->off_cat, pk->len_cat, Mt, Mt, Ll});
    } else {
      segs.push_back({0, B, pk->max_l, lig_mask});
      packs.push_back(AttnPack{pk->off_cat, pk->off_cat, pk->len_cat, Mt, Mt, Ll});
      segs.push_back({0, B, pk->max_r, rec_mask});
      packs.push_back(AttnPack{pk->off_cat + B, pk->off_cat + B, pk->len_cat + B, Mt, Mt, Lr});
    }
  } else if (Ll == Lr) {
    segs.push_back({0, 2 * B, Ll, f.maskcat});
  } else {
    segs.push_back({0, B, Ll, lig_mask});
    segs.push_back({Ml, B, Lr, rec_mask});
  }
  const int Lq_self = pl ? pl->max_l : Ll, Lk_cross = pk ? pk->max_r : Lr;
  const AttnPack* aps = pl ? &pk_self : nullptr;
  const AttnPack* apc = pk ? &pk_cross : nullptr;
  const SEHoist<T> hz_lig{Ml, inv ? inv->o : nullptr, inv ? inv->xr : nullptr, nullptr, nullptr};
  SD_TRY(se_layer<T>(*this, wfmt, se_lig, x, ccat, Mt, 1, Mt, segs, sb, x2, s, pl ? &packs : nullptr, nullptr, inv ? &hz_lig : nullptr));
  const T* rec = x2.t + MlH;

  // decoder: 6 x (self-attn -> cross-attn -> FFN), post-LN (HF BertLayer; model.py:226-231)
  SD_TRY(gemm_T(wfmt, Mr, NL * 2 * H, H, rec, ckv_all, ckv_all_b, 0, kv_all, s));
  Act<T> h = x2;  // ligand rows are the first Ml rows
  if constexpr (k16) {
    // 16-bit modes: a post-LN tensor h = LN(o) is needed (a) as the 16-bit A operand of the next GEMM and (b) in fp32 as the
    // residual of the GEMM after that.  (b) is rebuilt inside that GEMM's epilogue from the fp32 pre-LN tensor o, the per-row
    // (mean, rstd) the LN kernel emits and the LN affine -- the same fp32 formula, so bit-identical -- which lets the LN kernel
    // skip its 3 KB/row fp32 copy.  o needs three buffers with fixed roles (oA, oB, oC): every GEMM reads its residual from a
    // different buffer than the one it writes (attn_out: oC of the previous layer -> oA; cross_out: oA -> oB; ffn_down: oB -> oC).
    float* obuf[3] = {sb.o, sb.m2, f.obuf3};
    LnResid prev{};        // how to rebuild the current residual-stream value from `o_prev` (layer >= 1)
    const float* o_prev = nullptr;
    for (int i = 0; i < NL; ++i) {
      const LayerW& w = layers[i];
      const bool last = i + 1 == NL;
      const Act<T> h1 = hbuf[0], h2 = hbuf[1], h3 = hbuf[0];
      float* oA = obuf[0];
      float* oB = obuf[1];
      float* oC = obuf[2];
      SD_TRY(gemm_T(wfmt, Ml, 3 * H, H, h.t, w.self.qkv, w.self.qkv_b, 0, sb.qkv, s));
      SD_TRY(attention<T>(B, heads, Lq_self, Lq_self, sb.qkv, 3 * H, sb.qkv + H, 3 * H, sb.qkv + 2 * H, 3 * H, pick<T>(w.self.E), P, lig_mask, sb.ctx, s, aps));
      SD_TRY(gemm_ln<T>(wfmt, Ml, H, H, sb.ctx, w.self.out, w.self.out_b, i == 0 ? h.s : o_prev, oA, i == 0 ? nullptr : &prev, w.self.ln_w,
                        w.self.ln_b, eps, h1.t, lnstats, s));
      SD_TRY(gemm_T(wfmt, Ml, H, H, h1.t, w.cq, w.cq_b, 0, cq, s));
      const T* kbase = kv_all + static_cast<size_t>(i) * 2 * H;
      SD_TRY(attention<T>(B, heads, Lq_self, Lk_cross, cq, H, kbase, NL * 2 * H, kbase + H, NL * 2 * H, static_cast<const T*>(nullptr), P, rec_mask, sb.ctx, s, apc, K));
      const LnResid r1{lnstats, w.self.ln_w, w.self.ln_b};
      SD_TRY(gemm_ln<T>(wfmt, Ml, H, H, sb.ctx, w.cout, w.cout_b, oA, oB, &r1, w.cln_w, w.cln_b, eps, h2.t, lnstats + Ml, s));
      SD_TRY(gemm_T(wfmt, Ml, I, H, h2.t, w.inter, w.inter_b, 1, ffn, s));
      const LnResid r2{lnstats + Ml, w.cln_w, w.cln_b};
      if (last) {
        // the last layer's output feeds decoder_normalize, whose rowwise kernels read the fp32 stream: materialise it there
        SD_TRY(gemm_S(wfmt, Ml, H, I, ffn, w.outd, w.outd_b, oB, oC, s, &r2));
        SD_TRY(layernorm<T>(oC, Ml, H, w.oln_w, w.oln_b, eps, h3.s, h3.t, lnstats + 2 * static_cast<size_t>(Ml), s));
      } else {
        SD_TRY(gemm_ln<T>(wfmt, Ml, H, I, ffn, w.outd, w.outd_b, oB, oC, &r2, w.oln_w, w.oln_b, eps, h3.t, lnstats + 2 * static_cast<size_t>(Ml), s));
      }
      prev = LnResid{lnstats + 2 * static_cast<size_t>(Ml), w.oln_w, w.oln_b};
      o_prev = oC;
      h = h3;
    }
  } else {
    for (int i = 0; i < NL; ++i) {
      const LayerW& w = layers[i];
      // h is dead once the self-output GEMM has folded it in as the residual, so h1/h3 may reuse its buffer
      const Act<T> h1 = hbuf[0], h2 = hbuf[1], h3 = hbuf[0];
      SD_TRY(gemm_T(wfmt, Ml, 3 * H, H, h.t, w.self.qkv, w.self.qkv_b, 0, sb.qkv, s));
      SD_TRY(attention<T>(B, heads, Lq_self, Lq_self, sb.qkv, 3 * H, sb.qkv + H, 3 * H, sb.qkv + 2 * H, 3 * H, pick<T>(w.self.E), P, lig_mask, sb.ctx, s, aps));
      SD_TRY(gemm_S(wfmt, Ml, H, H, sb.ctx, w.self.out, w.self.out_b, h.s, sb.o, s));
      SD_TRY(layernorm<T>(sb.o, Ml, H, w.self.ln_w, w.self.ln_b, eps, h1.s, h1.t_out(), nullptr, s));
      SD_TRY(gemm_T(wfmt, Ml, H, H, h1.t, w.cq, w.cq_b, 0, cq, s));
      const T* kbase = kv_all + static_cast<size_t>(i) * 2 * H;
      SD_TRY(attention<T>(B, heads, Lq_self, Lk_cross, cq, H, kbase, NL * 2 * H, kbase + H, NL * 2 * H, static_cast<const T*>(nullptr), P, rec_mask, sb.ctx, s, apc, K));
      SD_TRY(gemm_S(wfmt, Ml, H, H, sb.ctx, w.cout, w.cout_b, h1.s, sb.o, s));
      SD_TRY(layernorm<T>(sb.o, Ml, H, w.cln_w, w.cln_b, eps, h2.s, h2.t_out(), nullptr, s));
      SD_TRY(gemm_T(wfmt, Ml, I, H, h2.t, w.inter, w.inter_b, 1, ffn, s));
      SD_TRY(gemm_S(wfmt, Ml, H, I, ffn, w.outd, w.outd_b, h2.s, sb.o, s));
      SD_TRY(layernorm<T>(sb.o, Ml, H, w.oln_w, w.oln_b, eps, h3.s, h3.t_out(), nullptr, s));
      h = h3;
    }
  }

  // decoder_normalize: SELayer conditioned on the timestep only (c broadcast over L; model.py:232-235).  Sampling loop: its
  // modulation is row *step_ptr of inv->mod.
  std::vector<Segment> lseg{{0, B, Lq_self, lig_mask}};
  std::vector<AttnPack> lpack;
  if (pl) lpack.push_back(pk_self);
  const SEHoist<T> hz_dec{Ml, nullptr, nullptr, inv ? static_cast<const T*>(inv->mod) : nullptr, step_ptr};
  SD_TRY(se_layer<T>(*this, wfmt, se_dec, h, teT, B, Ll, Ml, lseg, sb, x, s, pl ? &lpack : nullptr, pl ? pl->graph : nullptr, inv ? &hz_dec : nullptr));

  // AminoAcidPredictor (model.py:148-153)
  if constexpr (std::is_same<T, bf16>::value) {
    // bf16 mode: the output head runs on fp16 operands (same tensor-core rate).  Its input is the fp32 residual stream out of
    // decoder_normalize (bounded: LayerNorm-scale values), so fp16's 11-bit mantissa is safe and buys back the single most
    // sensitive rounding of the network: dense1's weights + its GELU output are 2 % of the FLOPs but ~15-20 % of the bf16 logit
    // error variance (profiles/bf16_attribution_r02.txt).  Everything upstream stays bf16.
    f16* xh = reinterpret_cast<f16*>(sb.ctx);  // free at this point: [Ml, H] 16-bit
    f16* yh = reinterpret_cast<f16*>(y);
    SD_TRY(f32_to_16<f16>(x.s, static_cast<size_t>(Ml) * H, xh, s));
    SD_TRY(gemm_16(Ml, H, H, xh, 0, p1.g, 0, p1_b, nullptr, 1, yh, 0, s));
    SD_TRY(predictor_tail<f16>(yh, Ml, H, p_ln_w, p_ln_b, 1e-12f, p2_w, p2_b, cfg.feature_size, logits, s, pl ? pl->src_l : nullptr));
    return SEQDIFF_OK;
  }
  SD_TRY(gemm_T(wfmt, Ml, H, H, x.t, p1, p1_b, 1, y, s));
  SD_TRY(predictor_tail<T>(y, Ml, H, p_ln_w, p_ln_b, 1e-12f, p2_w, p2_b, cfg.feature_size, logits, s, pl ? pl->src_l : nullptr));
  return SEQDIFF_OK;
}

int Model::forward(int precision, int B, int Ll, int Lr, const float* timestep, const int* step_ptr, const float* x_t,
                   const float* lig_angle, const float* lig_mask, const float* rec_seq_in, const float* rec_angle,
                   const float* rec_mask, float* logits, cudaStream_t s, const PackInfo* pk, const LoopInv* inv, int K) {
  SD_CHECK(finalized, "model not finalised (seqdiff_model_finalize)");
  SD_CHECK(arch == kArchSequence, "handle holds a structure model: use seqdiff_struct_forward");
  SD_CHECK(!pk || precision != SEQDIFF_FP32, "ragged packing runs in the 16-bit modes");
  SD_CHECK(precision >= SEQDIFF_FP32 && precision <= SEQDIFF_FP16, "unknown precision mode");
  SD_CHECK(B > 0 && Ll > 0 && Lr > 0, "empty batch");
  SD_CHECK(!inv || step_ptr, "the sampling-loop invariants are indexed by the device step counter");
  SD_CHECK(K >= 1 && B % K == 0 && (K == 1 || inv), "shared receptor rows (K > 1) exist in the sampling loop only");
  if (cfg.relative_key) SD_CHECK(Ll <= cfg.max_position_embeddings && Lr <= cfg.max_position_embeddings, "Length exceed");
  SD_CUDA(cudaSetDevice(device));
  SD_TRY(ensure_workspace(workspace_need(precision, B, Ll, Lr)));
  if (g_profiling) profile_mark("__begin__", s);  // host time between two calls is not the first kernel's
  const PdlScope pdl_scope(pdl_auto_mode(pk ? static_cast<long long>(pk->Ml) + pk->Mr : static_cast<long long>(B) * Ll + static_cast<long long>(B / K) * Lr));
  switch (precision) {
    case SEQDIFF_FP32:
      return forward_t<float>(1, B, Ll, Lr, timestep, step_ptr, x_t, lig_angle, lig_mask, rec_seq_in, rec_angle, rec_mask, logits, s, nullptr, inv, K);
    case SEQDIFF_BF16:
      return forward_t<bf16>(1, B, Ll, Lr, timestep, step_ptr, x_t, lig_angle, lig_mask, rec_seq_in, rec_angle, rec_mask, logits, s, pk, inv, K);
    default:  // SEQDIFF_FP16
      return forward_t<f16>(0, B, Ll, Lr, timestep, step_ptr, x_t, lig_angle, lig_mask, rec_seq_in, rec_angle, rec_mask, logits, s, pk, inv, K);
  }
}

// The per-sampling part of the loop (LoopInv): the kernels forward_t runs on the same inputs, so every value is the one the
// stand-alone forward computes at every step.  None of them splits K, so a GEMM row's result does not depend on M (T rows of steps
// here, B rows of one step there), and attention items are per (graph, head), so the receptor graphs give the same result without
// the ligand graphs next to them.  The receptor rows are those of the B / K pockets (forward_t's K).
template <typename T>
int Model::loop_invariants_t(int wfmt, int B, int K, int Ll, int Lr, int T_, const float* rec_seq_in, const float* rec_mask, const LoopInv& iv,
                             cudaStream_t s, const PackInfo* pk) {
  constexpr bool k16 = !std::is_same<T, float>::value;
  const int H = cfg.hidden_size, heads = cfg.num_attention_heads, P = cfg.max_position_embeddings;
  const int Pk = B / K;  // pockets
  const int Ml = pk ? pk->Ml : B * Ll, Mr = pk ? pk->Mr : Pk * Lr;
  const FwdBufs<T> f = carve_forward<T>(ws, s, B, H, cfg.intermediate_size, cfg.num_hidden_layers, B * Ll, Pk * Lr, Ml, Mr);
  // timestep features of steps 0 .. T-1 (row i: t = i, as (float)*step_ptr gives it) and decoder_normalize's adaLN GEMMs on them
  SD_TRY(timestep_embed(nullptr, nullptr, ts_W, T_, H, iv.te, k16 ? iv.teT : nullptr, Fmt<T>::v, s));
  SD_TRY(gemm_T(wfmt, T_, H, H, static_cast<const T*>(iv.teT), se_dec.ada0, se_dec.ada0_b, 2, static_cast<T*>(iv.u), s));
  SD_TRY(gemm_T(wfmt, T_, 6 * H, H, static_cast<const T*>(iv.u), se_dec.ada2, se_dec.ada2_b, 0, static_cast<T*>(iv.mod), s));
  // receptor sequence embedding
  EmbedJobs jobs{};
  jobs.n = 1;
  EmbedJob& jb = jobs.j[0];
  jb.x = rec_seq_in; jb.Wt = rec_seq.Wt_; jb.b = rec_seq.b; jb.lnw = rec_seq.ln_w; jb.lnb = rec_seq.ln_b;
  jb.out32 = iv.xr; jb.outT = k16 ? iv.xrT : nullptr; jb.M = Mr; jb.fin = rec_seq.fin; jb.L = Lr;
  if (pk) jb.src_rows = pk->src_r;
  SD_TRY(embed_ln_multi<T>(jobs, cfg.layer_norm_eps, H, s));
  // receptor rows of ligand_feature_emb's attention sublayer up to its output dense + residual (se_layer)
  const AttnW& a = se_lig.attn;
  T* qkv = f.sb.qkv;
  SD_TRY(gemm_T(wfmt, Mr, 3 * H, H, static_cast<const T*>(iv.xrT), a.qkv, a.qkv_b, 0, qkv, s));
  const AttnPack ap = pk ? AttnPack{pk->off_r, pk->off_r, pk->len_r, Mr, Mr, Lr} : AttnPack{};
  const int Lk = pk ? pk->max_r : Lr;
  SD_TRY(attention<T>(Pk, heads, Lk, Lk, qkv, 3 * H, qkv + H, 3 * H, qkv + 2 * H, 3 * H, pick<T>(a.E), P, rec_mask, f.sb.ctx, s, pk ? &ap : nullptr));
  SD_TRY(gemm_S(wfmt, Mr, H, H, f.sb.ctx, a.out, a.out_b, iv.xr, iv.o, s));
  return SEQDIFF_OK;
}

// =====================================================================================================
// reverse-diffusion loop: one captured CUDA graph per step shape, replayed T times
// =====================================================================================================
// Ragged packing: lengths from the (prefix-ones) masks, row maps, offsets.  *usable = false when a mask is not a prefix of ones
// (the caller then stays on the padded path) or a graph has no valid ligand / receptor token.  B ligand graphs, B / K pockets.
// lig_padded: every ligand length is Ll whatever the ligand mask says, so only the receptor masks are read and checked.
int Model::build_pack(int B, int K, int Ll, int Lr, const float* lig_mask, const float* rec_mask, cudaStream_t s, bool* usable,
                      bool lig_padded) {
  *usable = false;
  const int P = B / K;
  std::vector<float> hl(lig_padded ? 0 : static_cast<size_t>(B) * Ll), hr(static_cast<size_t>(P) * Lr);
  if (!lig_padded) SD_CUDA(cudaMemcpyAsync(hl.data(), lig_mask, hl.size() * 4, cudaMemcpyDefault, s));
  SD_CUDA(cudaMemcpyAsync(hr.data(), rec_mask, hr.size() * 4, cudaMemcpyDefault, s));
  SD_CUDA(cudaStreamSynchronize(s));
  std::vector<int> len_l(B, Ll), len_r(P);
  auto lengths = [&](const std::vector<float>& m, int G, int L, std::vector<int>& len) -> bool {
    for (int b = 0; b < G; ++b) {
      int n = 0;
      while (n < L && m[static_cast<size_t>(b) * L + n] == 1.0f) ++n;
      for (int i = n; i < L; ++i)
        if (m[static_cast<size_t>(b) * L + i] != 0.0f) return false;
      if (n == 0) return false;
      len[b] = n;
    }
    return true;
  };
  if ((!lig_padded && !lengths(hl, B, Ll, len_l)) || !lengths(hr, P, Lr, len_r)) return SEQDIFF_OK;
  int Ml = 0, Mr = 0, max_l = 0, max_r = 0;
  std::vector<int> off_l(B), off_r(P);
  for (int b = 0; b < B; ++b) {
    off_l[b] = Ml; Ml += len_l[b];
    max_l = len_l[b] > max_l ? len_l[b] : max_l;
  }
  for (int p = 0; p < P; ++p) {
    off_r[p] = Mr; Mr += len_r[p];
    max_r = len_r[p] > max_r ? len_r[p] : max_r;
  }
  // block layout (ints): src_l[Ml] | src_r[Mr] | graph[Ml+Mr] | off_l[B] | off_r[P] | len_l[B] | len_r[P] | off_cat[B+P] | len_cat[B+P]
  std::vector<int> blk;
  blk.reserve(2 * (static_cast<size_t>(Ml) + Mr) + 4 * (static_cast<size_t>(B) + P));
  for (int b = 0; b < B; ++b) for (int l = 0; l < len_l[b]; ++l) blk.push_back(b * Ll + l);
  for (int p = 0; p < P; ++p) for (int l = 0; l < len_r[p]; ++l) blk.push_back(p * Lr + l);
  for (int b = 0; b < B; ++b) for (int l = 0; l < len_l[b]; ++l) blk.push_back(b);
  for (int p = 0; p < P; ++p) for (int l = 0; l < len_r[p]; ++l) blk.push_back(p);
  for (int b = 0; b < B; ++b) blk.push_back(off_l[b]);
  for (int p = 0; p < P; ++p) blk.push_back(off_r[p]);
  for (int b = 0; b < B; ++b) blk.push_back(len_l[b]);
  for (int p = 0; p < P; ++p) blk.push_back(len_r[p]);
  for (int b = 0; b < B; ++b) blk.push_back(off_l[b]);
  for (int p = 0; p < P; ++p) blk.push_back(Ml + off_r[p]);
  for (int b = 0; b < B; ++b) blk.push_back(len_l[b]);
  for (int p = 0; p < P; ++p) blk.push_back(len_r[p]);
  // FNV-1a over K, the kind of pack and the block: a changed batch composition re-captures the step graph
  uint64_t hsh = 1469598103934665603ull;
  hsh ^= static_cast<uint32_t>(K); hsh *= 1099511628211ull;
  hsh ^= lig_padded ? 1u : 0u; hsh *= 1099511628211ull;
  for (int v : blk) { hsh ^= static_cast<uint32_t>(v); hsh *= 1099511628211ull; }
  bool fresh = false;
  if (blk.size() > pack_cap) {
    if (d_pack) { SD_CUDA(cudaDeviceSynchronize()); SD_CUDA(cudaFree(d_pack)); d_pack = nullptr; pack_cap = 0; }
    SD_CUDA(cudaMalloc(reinterpret_cast<void**>(&d_pack), blk.size() * sizeof(int)));
    pack_cap = blk.size();
    fresh = true;
  }
  if (fresh || hsh != pack.hash || pack.B != B || pack.P != P) {
    SD_CUDA(cudaMemcpyAsync(d_pack, blk.data(), blk.size() * sizeof(int), cudaMemcpyHostToDevice, s));
    SD_CUDA(cudaStreamSynchronize(s));  // blk is a stack-lifetime host buffer
  }
  PackInfo pi;
  pi.B = B; pi.P = P; pi.Ml = Ml; pi.Mr = Mr; pi.max_l = max_l; pi.max_r = max_r; pi.hash = hsh; pi.lig_padded = lig_padded;
  const int* p = d_pack;
  pi.src_l = p; p += Ml;
  pi.src_r = p; p += Mr;
  pi.graph = p; p += Ml + Mr;
  pi.off_l = p; p += B;
  pi.off_r = p; p += P;
  pi.len_l = p; p += B;
  pi.len_r = p; p += P;
  pi.off_cat = p; p += B + P;
  pi.len_cat = p;
  pack = pi;
  *usable = true;
  return SEQDIFF_OK;
}

int Model::loop_setup(int precision, int P, int K, int Ll, int Lr, int T, const float* q_tables, const float* x_in, const float* lig_angle,
                      const float* lig_mask, const float* rec_seq_in, const float* rec_angle, const float* rec_mask, cudaStream_t caller,
                      int flags, bool scoring, LoopIO* io, cudaStream_t* ls) {
  SD_CHECK(finalized, "model not finalised (seqdiff_model_finalize)");
  SD_CHECK(arch == kArchSequence, "handle holds a structure model: use seqdiff_struct_sample_multi / seqdiff_struct_score_multi");
  SD_CHECK(T >= 1 && P > 0 && K > 0 && Ll > 0 && Lr > 0, "bad sampling arguments");
  const int B = P * K;  // ligand graphs: sample j of pocket p is graph p * K + j
  SD_CHECK(cfg.feature_size == SEQDIFF_NUM_CLASSES, "sampling needs feature_size == 20");
  SD_CUDA(cudaSetDevice(device));  // before the stream / events are created: they belong to the handle's device
  if (!loop_stream) {
    SD_CUDA(cudaStreamCreateWithFlags(&loop_stream, cudaStreamNonBlocking));
    SD_CUDA(cudaEventCreateWithFlags(&ev_in, cudaEventDisableTiming));
    SD_CUDA(cudaEventCreateWithFlags(&ev_out, cudaEventDisableTiming));
  }
  // everything below runs on the private stream, ordered after the caller's prior work ...
  cudaStream_t s = loop_stream;
  *ls = s;
  SD_CUDA(cudaEventRecord(ev_in, caller));
  SD_CUDA(cudaStreamWaitEvent(s, ev_in, 0));
  const size_t Nl = static_cast<size_t>(B) * Ll, Nr = static_cast<size_t>(P) * Lr;
  // persistent inputs: x_cur | logits | lig_angle | lig_mask | rec_seq | rec_angle | rec_mask
  const size_t need_in = align256(Nl * 20 * 4) * 2 + align256(Nl * 8 * 4) + align256(Nl * 4) + align256(Nr * 20 * 4) +
                         align256(Nr * 8 * 4) + align256(Nr * 4);
  if (need_in + 16 * kGuardBytes > samp_in_bytes) {
    if (samp_in) { SD_CUDA(cudaDeviceSynchronize()); debug_guard_begin(samp_in); SD_CUDA(cudaFree(samp_in)); samp_in = nullptr; samp_in_bytes = 0; }
    SD_CUDA(cudaMalloc(reinterpret_cast<void**>(&samp_in), need_in + 16 * kGuardBytes));
    samp_in_bytes = need_in + 16 * kGuardBytes;
  }
  const size_t tab_floats = static_cast<size_t>(T) * 3 * 400;
  if (tab_floats > tables_cap) {
    if (d_tables) { SD_CUDA(cudaDeviceSynchronize()); SD_CUDA(cudaFree(d_tables)); d_tables = nullptr; tables_cap = 0; }
    SD_CUDA(cudaMalloc(reinterpret_cast<void**>(&d_tables), tab_floats * 4));
    tables_cap = tab_floats;
  }
  SD_TRY(ensure_workspace(workspace_need(precision, B, Ll, Lr)));
  Bump bp(samp_in, s);
  io->x_cur = bp.take<float>(Nl * 20);
  io->logits = bp.take<float>(Nl * 20);
  io->c_lang = bp.take<float>(Nl * 8);
  io->c_lmask = bp.take<float>(Nl);
  io->c_rseq = bp.take<float>(Nr * 20);
  io->c_rang = bp.take<float>(Nr * 8);
  io->c_rmask = bp.take<float>(Nr);
  if (scoring) {  // x0 | fp64 sums in a block of their own: scoring never moves the sampler's buffers (its cached graph stays valid)
    const size_t need_sc = align256(Nl * 20 * 4) + align256(Nl * 2 * 8) + 4 * kGuardBytes;
    if (need_sc > score_in_bytes) {
      if (score_in) { SD_CUDA(cudaDeviceSynchronize()); debug_guard_begin(score_in); SD_CUDA(cudaFree(score_in)); score_in = nullptr; score_in_bytes = 0; }
      SD_CUDA(cudaMalloc(reinterpret_cast<void**>(&score_in), need_sc));
      score_in_bytes = need_sc;
    }
    Bump bs(score_in, s);
    io->x0 = bs.take<float>(Nl * 20);
    io->acc = bs.take<double>(Nl * 2);
  }
  SD_CUDA(cudaMemcpyAsync(d_tables, q_tables, tab_floats * 4, cudaMemcpyDefault, s));
  SD_CUDA(cudaMemcpyAsync(scoring ? io->x0 : io->x_cur, x_in, Nl * 20 * 4, cudaMemcpyDefault, s));
  SD_CUDA(cudaMemcpyAsync(io->c_lang, lig_angle, Nl * 8 * 4, cudaMemcpyDefault, s));
  SD_CUDA(cudaMemcpyAsync(io->c_lmask, lig_mask, Nl * 4, cudaMemcpyDefault, s));
  SD_CUDA(cudaMemcpyAsync(io->c_rseq, rec_seq_in, Nr * 20 * 4, cudaMemcpyDefault, s));
  SD_CUDA(cudaMemcpyAsync(io->c_rang, rec_angle, Nr * 8 * 4, cudaMemcpyDefault, s));
  SD_CUDA(cudaMemcpyAsync(io->c_rmask, rec_mask, Nr * 4, cudaMemcpyDefault, s));
  if (scoring) SD_CUDA(cudaMemsetAsync(io->acc, 0, Nl * 2 * 8, s));
  // ragged packing (flags bit 0): valid prefixes only; needs the 16-bit kernels and prefix masks, otherwise the padded path runs
  const PackInfo* pk = nullptr;
  if ((flags & 1) && precision != SEQDIFF_FP32) {
    bool usable = false;
    SD_TRY(build_pack(B, K, Ll, Lr, io->c_lmask, io->c_rmask, s, &usable));
    if (usable) {
      pk = &pack;
      SD_CUDA(cudaMemsetAsync(io->logits, 0, Nl * 20 * 4, s));  // padded positions are never written in packed mode: defined as 0
    }
  }
  // padded path, 16-bit modes: the receptor rows are still packed (PackInfo::lig_padded), since no output reads a padded one.  It
  // needs prefix receptor masks with at least one valid token per pocket: a pocket without one attends uniformly over its padded
  // keys, whose values are then read.  Otherwise (and in fp32 mode) every receptor row is computed.
  if (!pk && precision != SEQDIFF_FP32) {
    bool usable = false;
    SD_TRY(build_pack(B, K, Ll, Lr, nullptr, io->c_rmask, s, &usable, true));
    if (usable) pk = &pack;
  }
  io->pk = pk;
  const long long rows = pk ? static_cast<long long>(pk->Ml) + pk->Mr : static_cast<long long>(Nl + Nr);  // token rows of a step
  io->rows = rows;
  // The per-sampling invariants (LoopInv), computed here by every call, outside the graph: the graph only holds their addresses.
  // Receptor rows first (P * Lr, the packed rows are a prefix), then the step tables with a grow-only capacity, so a cached graph
  // serves any T up to it.
  {
    inv.rows = T > inv.rows ? T : inv.rows;
    const size_t es = precision == SEQDIFF_FP32 ? 4 : 2, NrH = Nr * cfg.hidden_size, tH = static_cast<size_t>(inv.rows) * cfg.hidden_size;
    const size_t need_inv = 2 * align256(NrH * 4) + align256(NrH * 2) + align256(tH * 4) + align256(tH * 2) + align256(tH * es) +
                            align256(tH * 6 * es) + 8 * kGuardBytes;
    if (need_inv > samp_inv_bytes) {
      if (samp_inv) { SD_CUDA(cudaDeviceSynchronize()); debug_guard_begin(samp_inv); SD_CUDA(cudaFree(samp_inv)); samp_inv = nullptr; samp_inv_bytes = 0; }
      SD_CUDA(cudaMalloc(reinterpret_cast<void**>(&samp_inv), need_inv));
      samp_inv_bytes = need_inv;
    }
    Bump bi(samp_inv, s);
    inv.xr = bi.take<float>(NrH);
    inv.xrT = es == 2 ? static_cast<void*>(bi.take<uint16_t>(NrH)) : inv.xr;
    inv.o = bi.take<float>(NrH);
    inv.te = bi.take<float>(tH);
    inv.teT = es == 2 ? static_cast<void*>(bi.take<uint16_t>(tH)) : inv.te;
    inv.u = bi.take<uint8_t>(tH * es);
    inv.mod = bi.take<uint8_t>(tH * 6 * es);
    const PdlScope pdl_scope(pdl_auto_mode(rows));
    switch (precision) {
      case SEQDIFF_FP32: SD_TRY(loop_invariants_t<float>(1, B, K, Ll, Lr, T, io->c_rseq, io->c_rmask, inv, s, nullptr)); break;
      case SEQDIFF_BF16: SD_TRY(loop_invariants_t<bf16>(1, B, K, Ll, Lr, T, io->c_rseq, io->c_rmask, inv, s, pk)); break;
      default: SD_TRY(loop_invariants_t<f16>(0, B, K, Ll, Lr, T, io->c_rseq, io->c_rmask, inv, s, pk)); break;
    }
  }
  GraphKey& key = io->key;
  key.pack_hash = pk ? pk->hash : 0;
  key.precision = precision; key.B = B; key.K = K; key.Ll = Ll; key.Lr = Lr;
  key.ws_ptr = ws; key.in_ptr = samp_in; key.tab_ptr = d_tables;  // (seed, gid0) are NOT part of the key: device memory, see arm_loop_kernel
  key.inv_ptr = samp_inv; key.inv_rows = inv.rows;
  if (scoring) key.aux_ptr = score_in;
  return SEQDIFF_OK;
}

template <typename Fwd, typename Step>
int Model::replay_loop(cudaGraphExec_t& exec, GraphKey& cached, int& kernels, const GraphKey& key, int T, uint64_t seed, uint64_t gid0,
                       cudaStream_t s, const Fwd& fwd, const Step& step) {
  uint64_t* d_rng = reinterpret_cast<uint64_t*>(d_step + 16);
  if (!exec || !(key == cached)) {
    if (exec) { cudaGraphExecDestroy(exec); exec = nullptr; }
    // un-captured dry run of the forward: sets kernel attributes and fills the TMA descriptor cache
    SD_CUDA(launch_k(set_int_kernel, dim3(1), dim3(1), 0, s, d_step, T - 1));
    SD_LAUNCHED("set_int", s);
    SD_TRY(fwd(s));
    SD_CUDA(cudaStreamSynchronize(s));
    cudaGraph_t graph = nullptr;
    const uint64_t l0 = g_launches.load();
    SD_CUDA(cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal));
    const int rc = step(s);
    kernels = static_cast<int>(g_launches.load() - l0);  // kernel nodes per replay
    cudaError_t ce = cudaStreamEndCapture(s, &graph);
    if (rc != SEQDIFF_OK) { if (graph) cudaGraphDestroy(graph); return rc; }
    SD_CUDA(ce);
    ce = cudaGraphInstantiate(&exec, graph, 0);
    cudaGraphDestroy(graph);
    SD_CUDA(ce);
    cached = key;
  }
  SD_CUDA(launch_k(arm_loop_kernel, dim3(1), dim3(1), 0, s, d_step, T - 1, d_rng, seed, gid0));
  SD_LAUNCHED("arm_loop", s);
  for (int it = 0; it < T; ++it) SD_CUDA(cudaGraphLaunch(exec, s));
  g_launches.fetch_add(static_cast<uint64_t>(T) * kernels, std::memory_order_relaxed);  // replayed kernel nodes
  return SEQDIFF_OK;
}

int Model::sample(int precision, int P, int K, int Ll, int Lr, int T, const float* q_tables, const float* x_T, const float* lig_angle,
                  const float* lig_mask, const float* rec_seq_in, const float* rec_angle, const float* rec_mask, int diverse,
                  const float* noise_E, uint64_t seed, uint64_t gid0, float* final_out, cudaStream_t caller, int flags) {
  LoopIO io;
  cudaStream_t s = nullptr;
  SD_TRY(loop_setup(precision, P, K, Ll, Lr, T, q_tables, x_T, lig_angle, lig_mask, rec_seq_in, rec_angle, rec_mask, caller, flags, false, &io, &s));
  const int B = P * K;
  const PackInfo* pk = io.pk;
  GraphKey key = io.key;
  key.diverse = diverse; key.noise = noise_E;
  uint64_t* d_rng = reinterpret_cast<uint64_t*>(d_step + 16);
  auto fwd = [&](cudaStream_t st) -> int {
    return forward(precision, B, Ll, Lr, nullptr, d_step, io.x_cur, io.c_lang, io.c_lmask, io.c_rseq, io.c_rang, io.c_rmask, io.logits, st, pk, &inv, K);
  };
  auto one_step = [&](cudaStream_t st) -> int {
    const PdlScope pdl_scope(pdl_auto_mode(io.rows));
    SD_TRY(fwd(st));
    SD_TRY(reverse_step(d_tables, 1, B, Ll, io.x_cur, io.logits, diverse, noise_E, 0, 0, 0, d_step, io.x_cur, nullptr, st, d_step + 1, d_rng));
    return SEQDIFF_OK;
  };
  SD_TRY(replay_loop(graph_exec, graph_key, graph_kernels, key, T, seed, gid0, s, fwd, one_step));
  SD_CUDA(cudaMemcpyAsync(final_out, io.logits, static_cast<size_t>(B) * Ll * 20 * 4, cudaMemcpyDefault, s));
  // ... and the caller's stream continues only after the loop has finished
  SD_CUDA(cudaEventRecord(ev_out, s));
  SD_CUDA(cudaStreamWaitEvent(caller, ev_out, 0));
  return SEQDIFF_OK;
}

// One step of the score: x_t ~ q(x_t | x0) at the step's Qtb (the training q-sample), the sampling step's forward on it, then the
// step's bound terms (vlb_terms, which advances the step counter).  Same invariants, packing and K-per-pocket receptor rows as sample().
int Model::score(int precision, int P, int K, int Ll, int Lr, int T, const float* q_tables, const float* x0, const float* lig_angle,
                 const float* lig_mask, const float* rec_seq_in, const float* rec_angle, const float* rec_mask, const float* noise_E,
                 uint64_t seed, uint64_t gid0, double* terms_out, cudaStream_t caller, int flags) {
  LoopIO io;
  cudaStream_t s = nullptr;
  SD_TRY(loop_setup(precision, P, K, Ll, Lr, T, q_tables, x0, lig_angle, lig_mask, rec_seq_in, rec_angle, rec_mask, caller, flags, true, &io, &s));
  const int B = P * K;
  const PackInfo* pk = io.pk;
  GraphKey key = io.key;
  key.noise = noise_E;
  uint64_t* d_rng = reinterpret_cast<uint64_t*>(d_step + 16);
  auto fwd = [&](cudaStream_t st) -> int {
    return forward(precision, B, Ll, Lr, nullptr, d_step, io.x_cur, io.c_lang, io.c_lmask, io.c_rseq, io.c_rang, io.c_rmask, io.logits, st, pk, &inv, K);
  };
  auto one_step = [&](cudaStream_t st) -> int {
    const PdlScope pdl_scope(pdl_auto_mode(io.rows));
    SD_TRY(apply_aa_noise(d_tables, B, Ll, io.x0, noise_E, 0, 0, 0, io.x_cur, nullptr, st, d_step, d_rng));
    SD_TRY(fwd(st));
    SD_TRY(vlb_terms(d_tables, B, Ll, io.x0, io.x_cur, io.logits, io.c_lmask, d_step, d_step + 1, io.acc, st));
    return SEQDIFF_OK;
  };
  SD_TRY(replay_loop(score_exec, score_key, score_kernels, key, T, seed, gid0, s, fwd, one_step));
  SD_CUDA(cudaMemcpyAsync(terms_out, io.acc, static_cast<size_t>(B) * Ll * 2 * 8, cudaMemcpyDefault, s));
  SD_CUDA(cudaEventRecord(ev_out, s));
  SD_CUDA(cudaStreamWaitEvent(caller, ev_out, 0));
  return SEQDIFF_OK;
}

// =====================================================================================================
// structure (angle) model: structure_model/model.py:155-215 on the same kernels
// =====================================================================================================
// HF BertLayer, post-LN, fp32 residual stream: self-attention [-> cross-attention] -> FFN.  `o` is the fp32 pre-LN scratch,
// h1 / h2 the two rotating residual-stream tensors (h may be h1's buffer: it is dead once the self-output GEMM has folded it
// in).  Returns the buffer holding the layer output.
template <typename T>
static int bert_layer_plain(const Model& m, int wfmt, const LayerW& w, bool cross, int B, int Lq, int Lk, const Act<T>& h, const float* q_mask,
                            const float* k_mask, const T* kbase, int ldkv, T* qkv, T* ctx, T* cq, T* ffn, float* o, const Act<T>& h1,
                            const Act<T>& h2, Act<T>* out, cudaStream_t s, int kv_div = 1) {
  const int H = m.cfg.hidden_size, I = m.cfg.intermediate_size, heads = m.cfg.num_attention_heads, P = m.cfg.max_position_embeddings;
  const float eps = m.cfg.layer_norm_eps;
  const int M = B * Lq;
  SD_TRY(gemm_T(wfmt, M, 3 * H, H, h.t, w.self.qkv, w.self.qkv_b, 0, qkv, s));
  SD_TRY(attention<T>(B, heads, Lq, Lq, qkv, 3 * H, qkv + H, 3 * H, qkv + 2 * H, 3 * H, pick<T>(w.self.E), P, q_mask, ctx, s));
  SD_TRY(gemm_S(wfmt, M, H, H, ctx, w.self.out, w.self.out_b, h.s, o, s));
  SD_TRY(layernorm<T>(o, M, H, w.self.ln_w, w.self.ln_b, eps, h1.s, h1.t_out(), nullptr, s));
  Act<T> cur = h1, nxt = h2;
  if (cross) {
    SD_TRY(gemm_T(wfmt, M, H, H, h1.t, w.cq, w.cq_b, 0, cq, s));
    SD_TRY(attention<T>(B, heads, Lq, Lk, cq, H, kbase, ldkv, kbase + H, ldkv, static_cast<const T*>(nullptr), P, k_mask, ctx, s, nullptr, kv_div));
    SD_TRY(gemm_S(wfmt, M, H, H, ctx, w.cout, w.cout_b, h1.s, o, s));
    SD_TRY(layernorm<T>(o, M, H, w.cln_w, w.cln_b, eps, h2.s, h2.t_out(), nullptr, s));
    cur = h2;
    nxt = h1;
  }
  SD_TRY(gemm_T(wfmt, M, I, H, cur.t, w.inter, w.inter_b, 1, ffn, s));
  SD_TRY(gemm_S(wfmt, M, H, I, ffn, w.outd, w.outd_b, cur.s, o, s));
  SD_TRY(layernorm<T>(o, M, H, w.oln_w, w.oln_b, eps, nxt.s, nxt.t_out(), nullptr, s));
  *out = nxt;
  return SEQDIFF_OK;
}

// 16-bit modes: the same stack with the LayerNorm-rebuild flow of the sequence decoder (forward_t): a post-LN tensor exists only as
// the 16-bit operand of the next GEMM; its fp32 value, needed as the residual of the GEMM after that, is rebuilt in that GEMM's
// epilogue from the fp32 pre-LN tensor, the per-row (mean, rstd) and the affine -- the LayerNorm kernels skip their fp32 copy.
// Pre-LN buffers with fixed roles: obuf[0] self-output, obuf[1] cross-output, obuf[2] FFN-output (every GEMM reads its residual from
// a different buffer than the one it writes).  *out = 16-bit output of the last layer (all the consumers of a stack read).
// M token rows.  Ragged packing: aps / apc address the graphs of the self- / cross-attention (AttnPack), Lq / Lk are then the largest
// lengths and M the packed row count; without them M = B * Lq.  kv_div: query graph b cross-attends to key graph b / kv_div.
template <typename T>
static int bert_stack_lnresid(const Model& m, int wfmt, const std::vector<LayerW>& Ls, bool cross, int B, int Lq, int Lk, int M, const Act<T>& h0,
                              const float* q_mask, const float* k_mask, const T* kv_all, int ldkv, T* qkv, T* ctx, T* cq, T* ffn,
                              float* const (&obuf)[3], float2* lnstats, T* hT0, T* hT1, const T** out, cudaStream_t s,
                              const AttnPack* aps = nullptr, const AttnPack* apc = nullptr, int kv_div = 1) {
  const int H = m.cfg.hidden_size, I = m.cfg.intermediate_size, heads = m.cfg.num_attention_heads, P = m.cfg.max_position_embeddings;
  const float eps = m.cfg.layer_norm_eps;
  float2* stA = lnstats;
  float2* stB = lnstats + M;
  float2* stC = lnstats + 2 * static_cast<size_t>(M);
  LnResid prev{};
  const float* o_prev = nullptr;
  const T* h = h0.t;
  for (size_t i = 0; i < Ls.size(); ++i) {
    const LayerW& w = Ls[i];
    SD_TRY(gemm_T(wfmt, M, 3 * H, H, h, w.self.qkv, w.self.qkv_b, 0, qkv, s));
    SD_TRY(attention<T>(B, heads, Lq, Lq, qkv, 3 * H, qkv + H, 3 * H, qkv + 2 * H, 3 * H, pick<T>(w.self.E), P, q_mask, ctx, s, aps));
    SD_TRY(gemm_ln<T>(wfmt, M, H, H, ctx, w.self.out, w.self.out_b, i == 0 ? h0.s : o_prev, obuf[0], i == 0 ? nullptr : &prev, w.self.ln_w,
                      w.self.ln_b, eps, hT0, stA, s));
    const T* cur = hT0;
    const float* o_cur = obuf[0];
    LnResid rc{stA, w.self.ln_w, w.self.ln_b};
    if (cross) {
      SD_TRY(gemm_T(wfmt, M, H, H, hT0, w.cq, w.cq_b, 0, cq, s));
      const T* kbase = kv_all + i * 2 * static_cast<size_t>(H);
      SD_TRY(attention<T>(B, heads, Lq, Lk, cq, H, kbase, ldkv, kbase + H, ldkv, static_cast<const T*>(nullptr), P, k_mask, ctx, s, apc, kv_div));
      SD_TRY(gemm_ln<T>(wfmt, M, H, H, ctx, w.cout, w.cout_b, obuf[0], obuf[1], &rc, w.cln_w, w.cln_b, eps, hT1, stB, s));
      cur = hT1;
      o_cur = obuf[1];
      rc = LnResid{stB, w.cln_w, w.cln_b};
    }
    SD_TRY(gemm_T(wfmt, M, I, H, cur, w.inter, w.inter_b, 1, ffn, s));
    T* nxt = cross ? hT0 : hT1;
    SD_TRY(gemm_ln<T>(wfmt, M, H, I, ffn, w.outd, w.outd_b, o_cur, obuf[2], &rc, w.oln_w, w.oln_b, eps, nxt, stC, s));
    prev = LnResid{stC, w.oln_w, w.oln_b};
    o_prev = obuf[2];
    h = nxt;
  }
  *out = h;
  return SEQDIFF_OK;
}

size_t Model::struct_workspace_need(int precision, int B, int Ll, int Lr, int K) const {
  const size_t es = precision == SEQDIFF_FP32 ? 4 : 2;
  const size_t H = cfg.hidden_size, I = cfg.intermediate_size, NL = cfg.num_hidden_layers;
  const size_t Ml = static_cast<size_t>(B) * Ll, Mr = static_cast<size_t>(B / K) * Lr, Mx = Ml > Mr ? Ml : Mr;
  size_t n = align256(Mr * NL * 2 * H * es);           // cross K|V of every decoder layer: survives between forwards
  n += 2 * align256(static_cast<size_t>(B) * H * 4);   // te fp32 + operand copy
  n += 5 * (align256(Mx * H * 4) + align256(Mx * H * 2));  // x, x2, x1, h ping-pong (stream + operand)
  n += 2 * align256(Mx * H * 4);                       // o, m2
  n += 5 * align256(Mx * H * es);                      // c, u, ctx, cq, y
  n += align256(Mx * 6 * H * es) + align256(Mx * 3 * H * es) + align256(Mx * 4 * H * es);  // mod, qkv, m1
  n += align256(Mx * I * es);                          // ffn
  return n + 8192 + 64 * kGuardBytes;  // (debug build: one guard band per carved buffer)
}

template <typename T>
int Model::struct_forward_t(int wfmt, int B, int Ll, int Lr, const float* timestep, const int* step_ptr, const float* noised,
                            const float* lig_mask, const float* rec_seq_in, const float* rec_angle, const float* rec_mask, float* out,
                            int phases, cudaStream_t s, const PackInfo* pk, int K) {
  constexpr bool k16 = !std::is_same<T, float>::value;
  const int H = cfg.hidden_size, I = cfg.intermediate_size, NL = cfg.num_hidden_layers;
  const float eps = cfg.layer_norm_eps;
  // packed (ragged) batch: only the valid prefix of every graph is a row; the buffers keep their padded sizes, inputs, masks and
  // the output their padded layouts.  The receptor side holds the B / K pockets: ligand graph b reads pocket b / K.
  const int Pk = B / K;
  const int Mlp = B * Ll, Mrp = Pk * Lr, Mx = Mlp > Mrp ? Mlp : Mrp;
  const int Ml = pk ? pk->Ml : Mlp, Mr = pk ? pk->Mr : Mrp;
  const int Lq = pk ? pk->max_l : Ll, Lk = pk ? pk->max_r : Lr;  // attention: largest ligand / receptor length
  AttnPack ap_l{}, ap_r{}, ap_x{};
  if (pk) {
    ap_l = AttnPack{pk->off_l, pk->off_l, pk->len_l, Ml, Ml, Ll};
    ap_r = AttnPack{pk->off_r, pk->off_r, pk->len_r, Mr, Mr, Lr};
    ap_x = AttnPack{pk->off_l, pk->off_r, pk->len_l, Ml, Mr, Lr};
  }
  const size_t MxH = static_cast<size_t>(Mx) * H;
  Bump bp(ws, s);
  T* kv_all = bp.take<T>(static_cast<size_t>(Mrp) * NL * 2 * H);  // first: same address for every (B, Ll, Lr) of a loop
  float* te = bp.take<float>(static_cast<size_t>(B) * H);
  T* teT = k16 ? bp.take<T>(static_cast<size_t>(B) * H) : reinterpret_cast<T*>(te);
  Act<T> x = take_act<T>(bp, MxH);
  Act<T> x2 = take_act<T>(bp, MxH);
  SEBufs<T> sb;
  sb.x1 = take_act<T>(bp, MxH);
  Act<T> hb[2] = {take_act<T>(bp, MxH), take_act<T>(bp, MxH)};
  sb.o = bp.take<float>(MxH);
  sb.m2 = bp.take<float>(MxH);
  T* cT = bp.take<T>(MxH);
  sb.u = bp.take<T>(MxH);
  sb.ctx = bp.take<T>(MxH);
  T* cq = bp.take<T>(MxH);
  T* y = bp.take<T>(MxH);
  sb.mod = bp.take<T>(MxH * 6);
  sb.qkv = bp.take<T>(MxH * 3);
  sb.m1 = bp.take<T>(MxH * 4);
  T* ffn = bp.take<T>(static_cast<size_t>(Mx) * I);
  auto job = [&](const float* in, int M, const EmbW& e, int L, float* o32, T* oT, bool lig) {
    EmbedJob jb{};
    jb.x = in; jb.Wt = e.Wt_; jb.b = e.b; jb.lnw = e.ln_w; jb.lnb = e.ln_b; jb.te = nullptr;
    jb.out32 = o32; jb.outT = oT; jb.M = M; jb.fin = e.fin; jb.L = L;
    if (pk) {
      jb.src_rows = lig ? pk->src_l : pk->src_r;
      jb.row_graph = lig ? pk->graph : pk->graph + pk->Ml;
    }
    return jb;
  };

  if (phases & 1) {
    // receptor branch (model.py:192-202): x = LN(Linear(angles)), c = LN(Linear(seq)); receptor_emb; 12 x (self-attn, FFN)
    EmbedJobs jobs{};
    jobs.n = 2;
    jobs.j[0] = job(rec_angle, Mr, rec_ang, Lr, x.s, x.t_out(), false);
    jobs.j[1] = job(rec_seq_in, Mr, rec_seq, Lr, k16 ? nullptr : reinterpret_cast<float*>(cT), k16 ? cT : nullptr, false);
    SD_TRY(embed_ln_multi<T>(jobs, eps, H, s));
    std::vector<Segment> rseg{{0, Pk, Lk, rec_mask}};
    const std::vector<AttnPack> rpack{ap_r};
    SD_TRY(se_layer<T>(*this, wfmt, se_lig, x, cT, Mr, 1, Mr, rseg, sb, x2, s, pk ? &rpack : nullptr));
    const T* enc_out = nullptr;
    if constexpr (k16) {
      float* const obuf[3] = {sb.o, sb.m2, hb[0].s};
      SD_TRY(bert_stack_lnresid<T>(*this, wfmt, enc_layers, false, Pk, Lk, Lk, Mr, x2, rec_mask, nullptr, nullptr, 0, sb.qkv, sb.ctx, cq, ffn, obuf,
                                   reinterpret_cast<float2*>(hb[1].s), hb[0].t, hb[1].t, &enc_out, s, pk ? &ap_r : nullptr));
    } else {
      Act<T> h = x2;
      for (int i = 0; i < NL; ++i) {
        Act<T> nh;
        SD_TRY(bert_layer_plain<T>(*this, wfmt, enc_layers[i], false, Pk, Lr, Lr, h, rec_mask, nullptr, nullptr, 0, sb.qkv, sb.ctx, cq, ffn, sb.o,
                                   hb[0], hb[1], &nh, s));
        h = nh;
      }
      enc_out = h.t;
    }
    // every decoder layer's cross K|V in one GEMM: the only thing the decoder reads from the receptor side
    SD_TRY(gemm_T(wfmt, Mr, NL * 2 * H, H, enc_out, ckv_all, ckv_all_b, 0, kv_all, s));
  }

  if (!(phases & 2)) return SEQDIFF_OK;
  // ligand branch (model.py:203-215)
  SD_TRY(timestep_embed(timestep, step_ptr, ts_W, B, H, te, k16 ? static_cast<void*>(teT) : nullptr, Fmt<T>::v, s));
  {
    EmbedJobs jobs{};
    jobs.n = 1;
    jobs.j[0] = job(noised, Ml, lig_ang, Ll, x.s, x.t_out(), true);
    SD_TRY(embed_ln_multi<T>(jobs, eps, H, s));
  }
  // timestep_emb: c broadcast over L (packed: every row takes the timestep features of its graph)
  std::vector<Segment> lseg{{0, B, Lq, lig_mask}};
  const std::vector<AttnPack> lpack{ap_l};
  SD_TRY(se_layer<T>(*this, wfmt, se_dec, x, teT, B, Ll, Ml, lseg, sb, x2, s, pk ? &lpack : nullptr, pk ? pk->graph : nullptr));
  const T* dec_out = nullptr;
  if constexpr (k16) {
    float* const obuf[3] = {sb.o, sb.m2, hb[0].s};
    SD_TRY(bert_stack_lnresid<T>(*this, wfmt, layers, true, B, Lq, Lk, Ml, x2, lig_mask, rec_mask, kv_all, NL * 2 * H, sb.qkv, sb.ctx, cq, ffn, obuf,
                                 reinterpret_cast<float2*>(hb[1].s), hb[0].t, hb[1].t, &dec_out, s, pk ? &ap_l : nullptr, pk ? &ap_x : nullptr, K));
  } else {
    Act<T> h = x2;
    for (int i = 0; i < NL; ++i) {
      Act<T> nh;
      const T* kbase = kv_all + static_cast<size_t>(i) * 2 * H;
      SD_TRY(bert_layer_plain<T>(*this, wfmt, layers[i], true, B, Ll, Lr, h, lig_mask, rec_mask, kbase, NL * 2 * H, sb.qkv, sb.ctx, cq, ffn, sb.o,
                                 hb[0], hb[1], &nh, s, K));
      h = nh;
    }
    dec_out = h.t;
  }
  SD_TRY(gemm_T(wfmt, Ml, H, H, dec_out, p1, p1_b, 1, y, s));
  SD_TRY(predictor_tail<T>(y, Ml, H, p_ln_w, p_ln_b, 1e-12f, p2_w, p2_b, cfg.feature_size, out, s, pk ? pk->src_l : nullptr));
  return SEQDIFF_OK;
}

int Model::struct_forward(int precision, int B, int Ll, int Lr, const float* timestep, const int* step_ptr, const float* noised,
                          const float* lig_mask, const float* rec_seq_in, const float* rec_angle, const float* rec_mask, float* out,
                          int phases, cudaStream_t s, const PackInfo* pk, int K) {
  SD_CHECK(finalized, "model not finalised (seqdiff_model_finalize)");
  SD_CHECK(arch == kArchStructure, "handle holds a sequence model: use seqdiff_forward");
  const PdlScope pdl_on(3);  // launch-bound path: programmatic dependent launch of the heavy kernels (42.3 -> 43.0 k graph-steps/s against every launch)
  SD_CHECK(precision >= SEQDIFF_FP32 && precision <= SEQDIFF_FP16, "unknown precision mode");
  SD_CHECK(!pk || precision != SEQDIFF_FP32, "ragged packing runs in the 16-bit modes");
  SD_CHECK(B > 0 && Ll > 0 && Lr > 0, "empty batch");
  SD_CHECK(K >= 1 && B % K == 0, "every pocket must serve K whole ligand graphs");
  if (cfg.relative_key) SD_CHECK(Ll <= cfg.max_position_embeddings && Lr <= cfg.max_position_embeddings, "Length exceed");
  SD_CUDA(cudaSetDevice(device));
  SD_TRY(ensure_workspace(struct_workspace_need(precision, B, Ll, Lr, K)));
  if (g_profiling) profile_mark("__begin__", s);
  switch (precision) {
    case SEQDIFF_FP32:
      return struct_forward_t<float>(1, B, Ll, Lr, timestep, step_ptr, noised, lig_mask, rec_seq_in, rec_angle, rec_mask, out, phases, s, nullptr, K);
    case SEQDIFF_BF16:
      return struct_forward_t<bf16>(1, B, Ll, Lr, timestep, step_ptr, noised, lig_mask, rec_seq_in, rec_angle, rec_mask, out, phases, s, pk, K);
    default:
      return struct_forward_t<f16>(0, B, Ll, Lr, timestep, step_ptr, noised, lig_mask, rec_seq_in, rec_angle, rec_mask, out, phases, s, pk, K);
  }
}

int Model::struct_loop_setup(int precision, int P, int K, int Ll, int Lr, int T, const float* table, const float* x_in, const float* lig_mask,
                             const float* rec_seq_in, const float* rec_angle, const float* rec_mask, cudaStream_t caller, int flags,
                             bool scoring, StructIO* io, cudaStream_t* ls) {
  SD_CHECK(finalized, "model not finalised (seqdiff_model_finalize)");
  SD_CHECK(arch == kArchStructure, scoring ? "handle holds a sequence model: use seqdiff_score_multi" : "handle holds a sequence model: use seqdiff_sample");
  SD_CHECK(T >= 1 && P > 0 && K > 0 && Ll > 0 && Lr > 0, "bad sampling arguments");
  const int B = P * K;  // ligand graphs: sample j of pocket p is graph p * K + j
  SD_CUDA(cudaSetDevice(device));
  if (!loop_stream) {
    SD_CUDA(cudaStreamCreateWithFlags(&loop_stream, cudaStreamNonBlocking));
    SD_CUDA(cudaEventCreateWithFlags(&ev_in, cudaEventDisableTiming));
    SD_CUDA(cudaEventCreateWithFlags(&ev_out, cudaEventDisableTiming));
  }
  // everything below runs on the private stream, ordered after the caller's prior work
  cudaStream_t s = loop_stream;
  *ls = s;
  SD_CUDA(cudaEventRecord(ev_in, caller));
  SD_CUDA(cudaStreamWaitEvent(s, ev_in, 0));
  const int F = cfg.feature_size;
  const size_t Nl = static_cast<size_t>(B) * Ll, Nr = static_cast<size_t>(P) * Lr;
  // persistent inputs: x_cur | model_out | lig_mask | rec_seq | rec_angle | rec_mask
  const size_t need_in = align256(Nl * F * 4) * 2 + align256(Nl * 4) + align256(Nr * 20 * 4) + align256(Nr * F * 4) + align256(Nr * 4);
  if (need_in + 16 * kGuardBytes > samp_in_bytes) {
    if (samp_in) { SD_CUDA(cudaDeviceSynchronize()); debug_guard_begin(samp_in); SD_CUDA(cudaFree(samp_in)); samp_in = nullptr; samp_in_bytes = 0; }
    SD_CUDA(cudaMalloc(reinterpret_cast<void**>(&samp_in), need_in + 16 * kGuardBytes));
    samp_in_bytes = need_in + 16 * kGuardBytes;
  }
  const size_t tab_floats = static_cast<size_t>(T) * (scoring ? 2 : 4);
  if (!scoring && tab_floats > tables_cap) {
    if (d_tables) { SD_CUDA(cudaDeviceSynchronize()); SD_CUDA(cudaFree(d_tables)); d_tables = nullptr; tables_cap = 0; }
    SD_CUDA(cudaMalloc(reinterpret_cast<void**>(&d_tables), tab_floats * 4));
    tables_cap = tab_floats;
  }
  SD_TRY(ensure_workspace(struct_workspace_need(precision, B, Ll, Lr, K)));
  Bump bp(samp_in, s);
  io->x_cur = bp.take<float>(Nl * F);
  io->mout = bp.take<float>(Nl * F);
  io->c_lmask = bp.take<float>(Nl);
  io->c_rseq = bp.take<float>(Nr * 20);
  io->c_rang = bp.take<float>(Nr * F);
  io->c_rmask = bp.take<float>(Nr);
  // x0 | fp64 sums | q-sample table in a block of their own: scoring never moves the sampler's buffers (its cached graph stays valid).
  // The table goes last, so the addresses the score's step graph holds depend on (B, Ll) and the block's base only, all in its key: a
  // cached graph serves any T, and the kernels read the step from the device counter.
  if (scoring) {
    const size_t need_sc = align256(Nl * F * 4) + align256(Nl * F * 8) + align256(tab_floats * 4) + 4 * kGuardBytes;
    if (need_sc > score_in_bytes) {
      if (score_in) { SD_CUDA(cudaDeviceSynchronize()); debug_guard_begin(score_in); SD_CUDA(cudaFree(score_in)); score_in = nullptr; score_in_bytes = 0; }
      SD_CUDA(cudaMalloc(reinterpret_cast<void**>(&score_in), need_sc));
      score_in_bytes = need_sc;
    }
    Bump bs(score_in, s);
    io->x0 = bs.take<float>(Nl * F);
    io->acc = bs.take<double>(Nl * F);
    io->qs = bs.take<float>(tab_floats);
  }
  SD_CUDA(cudaMemcpyAsync(scoring ? io->qs : d_tables, table, tab_floats * 4, cudaMemcpyDefault, s));
  // scoring: x_cur starts as x0 too, so that the un-captured dry run of the ligand branch reads defined angles
  SD_CUDA(cudaMemcpyAsync(io->x_cur, x_in, Nl * F * 4, cudaMemcpyDefault, s));
  if (scoring) SD_CUDA(cudaMemcpyAsync(io->x0, x_in, Nl * F * 4, cudaMemcpyDefault, s));
  SD_CUDA(cudaMemcpyAsync(io->c_lmask, lig_mask, Nl * 4, cudaMemcpyDefault, s));
  SD_CUDA(cudaMemcpyAsync(io->c_rseq, rec_seq_in, Nr * 20 * 4, cudaMemcpyDefault, s));
  SD_CUDA(cudaMemcpyAsync(io->c_rang, rec_angle, Nr * F * 4, cudaMemcpyDefault, s));
  SD_CUDA(cudaMemcpyAsync(io->c_rmask, rec_mask, Nr * 4, cudaMemcpyDefault, s));
  if (scoring) SD_CUDA(cudaMemsetAsync(io->acc, 0, Nl * F * 8, s));
  // ragged packing (flags bit 0): valid prefixes only, ligand offsets per sample and receptor offsets per pocket; needs the 16-bit
  // kernels and prefix masks with a valid position in every complex, otherwise the padded path runs.
  const PackInfo* pk = nullptr;
  if ((flags & 1) && precision != SEQDIFF_FP32) {
    bool usable = false;
    SD_TRY(build_pack(B, K, Ll, Lr, io->c_lmask, io->c_rmask, s, &usable));
    if (usable) pk = &pack;
  }
  io->pk = pk;
  GraphKey& key = io->key;
  key.pack_hash = pk ? pk->hash : 0;
  key.precision = precision; key.B = B; key.K = K; key.Ll = Ll; key.Lr = Lr; key.diverse = 0;
  key.ws_ptr = ws; key.in_ptr = samp_in;  // (seed, gid0) are NOT part of the key: device memory, see arm_loop_kernel
  if (scoring) key.aux_ptr = score_in;
  else key.tab_ptr = d_tables;
  return SEQDIFF_OK;
}

template <typename Step>
int Model::struct_replay(cudaGraphExec_t& exec, GraphKey& cached, int& kernels, const GraphKey& key, int precision, int K, int Ll, int Lr, int T,
                         uint64_t seed, uint64_t gid0, const StructIO& io, cudaStream_t s, const Step& step) {
  uint64_t* d_rng = reinterpret_cast<uint64_t*>(d_step + 16);
  // receptor branch once, eagerly (also the un-captured dry run that sets kernel attributes and fills the TMA descriptor cache)
  SD_CUDA(launch_k(arm_loop_kernel, dim3(1), dim3(1), 0, s, d_step, T - 1, d_rng, seed, gid0));
  SD_LAUNCHED("arm_loop", s);
  const bool hit = exec && key == cached;
  SD_TRY(struct_forward(precision, key.B, Ll, Lr, nullptr, d_step, io.x_cur, io.c_lmask, io.c_rseq, io.c_rang, io.c_rmask, io.mout, hit ? 1 : 3, s,
                        io.pk, K));
  if (!hit) {
    if (exec) { cudaGraphExecDestroy(exec); exec = nullptr; }
    SD_CUDA(cudaStreamSynchronize(s));
    cudaGraph_t graph = nullptr;
    const uint64_t l0 = g_launches.load();
    SD_CUDA(cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal));
    const int rc = step(s);
    kernels = static_cast<int>(g_launches.load() - l0);  // kernel nodes per replay
    cudaError_t ce = cudaStreamEndCapture(s, &graph);
    if (rc != SEQDIFF_OK) { if (graph) cudaGraphDestroy(graph); return rc; }
    SD_CUDA(ce);
    ce = cudaGraphInstantiate(&exec, graph, 0);
    cudaGraphDestroy(graph);
    SD_CUDA(ce);
    cached = key;
  }
  for (int it = 0; it < T; ++it) SD_CUDA(cudaGraphLaunch(exec, s));
  g_launches.fetch_add(static_cast<uint64_t>(T) * kernels, std::memory_order_relaxed);  // replayed kernel nodes
  return SEQDIFF_OK;
}

// structure_model/sample.py:104-144.  The receptor branch runs ONCE (it sees neither t nor the ligand; the reference recomputes
// it every step) and over the P pockets only; each step replays one captured graph: ligand branch + Gaussian reverse step + wrap.
int Model::struct_sample(int precision, int P, int K, int Ll, int Lr, int T, const float* coef_steps, const float* x_T, const float* lig_mask,
                         const float* rec_seq_in, const float* rec_angle, const float* rec_mask, const float* noise_steps, uint64_t seed,
                         uint64_t gid0, float* steps_out, float* final_out, cudaStream_t caller, int flags) {
  const PdlScope pdl_on(3);
  StructIO io;
  cudaStream_t s = nullptr;
  SD_TRY(struct_loop_setup(precision, P, K, Ll, Lr, T, coef_steps, x_T, lig_mask, rec_seq_in, rec_angle, rec_mask, caller, flags, false, &io, &s));
  const int B = P * K, F = cfg.feature_size;
  const PackInfo* pk = io.pk;
  GraphKey key = io.key;
  key.noise = noise_steps; key.aux_ptr = steps_out; key.T = T;
  uint64_t* d_rng = reinterpret_cast<uint64_t*>(d_step + 16);
  // the Gaussian step writes the padded positions of x_cur and steps_out as 0 in packed mode
  auto one_step = [&](cudaStream_t st) -> int {
    SD_TRY(struct_forward(precision, B, Ll, Lr, nullptr, d_step, io.x_cur, io.c_lmask, io.c_rseq, io.c_rang, io.c_rmask, io.mout, 2, st, pk, K));
    SD_TRY(gauss_step(d_tables, T, B, Ll * F, io.x_cur, io.mout, noise_steps, 0, 0, 0, d_step, io.x_cur, steps_out, st, d_step + 1, true, d_rng,
                      pk ? pk->len_l : nullptr, F));
    return SEQDIFF_OK;
  };
  SD_TRY(struct_replay(graph_exec, graph_key, graph_kernels, key, precision, K, Ll, Lr, T, seed, gid0, io, s, one_step));
  SD_CUDA(cudaMemcpyAsync(final_out, io.x_cur, static_cast<size_t>(B) * Ll * F * 4, cudaMemcpyDefault, s));
  // ... and the caller's stream continues only after the loop has finished
  SD_CUDA(cudaEventRecord(ev_out, s));
  SD_CUDA(cudaStreamWaitEvent(caller, ev_out, 0));
  return SEQDIFF_OK;
}

// Backbone score: one step is the training q-sample of x0 at step k (angle_qsample), the sampler's ligand branch at timestep k on it,
// then the step's objective terms (angle_score_terms, which advances the step counter).  Same staging, packing, K-per-pocket receptor
// rows and eager receptor branch as struct_sample(), but its own graph, key and input block.
int Model::struct_score(int precision, int P, int K, int Ll, int Lr, int T, const float* qs_steps, const float* x0, const float* lig_mask,
                        const float* rec_seq_in, const float* rec_angle, const float* rec_mask, const float* noise_steps, uint64_t seed,
                        uint64_t gid0, double* terms_out, cudaStream_t caller, int flags) {
  const PdlScope pdl_on(3);
  StructIO io;
  cudaStream_t s = nullptr;
  SD_TRY(struct_loop_setup(precision, P, K, Ll, Lr, T, qs_steps, x0, lig_mask, rec_seq_in, rec_angle, rec_mask, caller, flags, true, &io, &s));
  const int B = P * K, F = cfg.feature_size;
  const PackInfo* pk = io.pk;
  GraphKey key = io.key;
  key.noise = noise_steps;
  uint64_t* d_rng = reinterpret_cast<uint64_t*>(d_step + 16);
  auto one_step = [&](cudaStream_t st) -> int {
    SD_TRY(angle_qsample(io.qs, B, Ll * F, io.x0, noise_steps, d_step, d_rng, io.x_cur, st, pk ? pk->len_l : nullptr, F));
    SD_TRY(struct_forward(precision, B, Ll, Lr, nullptr, d_step, io.x_cur, io.c_lmask, io.c_rseq, io.c_rang, io.c_rmask, io.mout, 2, st, pk, K));
    SD_TRY(angle_score_terms(B, Ll * F, io.mout, noise_steps, io.c_lmask, d_step, d_step + 1, d_rng, io.acc, st, pk ? pk->len_l : nullptr, F));
    return SEQDIFF_OK;
  };
  SD_TRY(struct_replay(score_exec, score_key, score_kernels, key, precision, K, Ll, Lr, T, seed, gid0, io, s, one_step));
  SD_CUDA(cudaMemcpyAsync(terms_out, io.acc, static_cast<size_t>(B) * Ll * F * 8, cudaMemcpyDefault, s));
  SD_CUDA(cudaEventRecord(ev_out, s));
  SD_CUDA(cudaStreamWaitEvent(caller, ev_out, 0));
  return SEQDIFF_OK;
}

}  // namespace seqdiff
