// rowwise.cu -- the HBM-bound per-token kernels of the denoiser: timestep features, BertEmbeddings
// (Linear + LayerNorm), post-LN, the SELayer adaLN residual update, and the predictor tail.
// One warp owns one token row (H = 256*VPL features, 8 contiguous elements per lane per vector => 16 B
// (bf16) / 32 B (f32) per lane, fully coalesced); LayerNorm statistics are always fp32, two-pass
// (mean, then centred variance) like ATen's CPU kernel.
#include <cstdlib>

#include "common.cuh"
#include "kernels.h"

namespace seqdiff {

constexpr int kRowThreads = 256;  // 8 warps = 8 rows per CTA
constexpr int kEmbedTok = 2;     // tokens per warp pass of the embedding kernel (2: ~100 registers, two CTAs per SM)

template <typename T, int VPL>
__device__ __forceinline__ void load_row(const T* __restrict__ row, int lane, float (&v)[VPL][8]) {
#pragma unroll
  for (int i = 0; i < VPL; ++i) load8<T>(row + (i * 32 + lane) * 8, v[i]);
}
template <typename T, int VPL>
__device__ __forceinline__ void store_row(T* __restrict__ row, int lane, const float (&v)[VPL][8]) {
#pragma unroll
  for (int i = 0; i < VPL; ++i) store8<T>(row + (i * 32 + lane) * 8, v[i]);
}
template <int VPL>
__device__ __forceinline__ void row_stats(const float (&v)[VPL][8], int H, float eps, float& mean, float& rstd) {
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < VPL; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) s += v[i][j];
  mean = warp_sum(s) / static_cast<float>(H);
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < VPL; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float d = v[i][j] - mean;
      q = fmaf(d, d, q);
    }
  const float var = warp_sum(q) / static_cast<float>(H);
  rstd = 1.0f / sqrtf(var + eps);
}

// ---------------------------------------------------------------------------------------------------
// out16 (optional): the same values in the 16-bit operand format (fmt16: 0 = fp16, 1 = bf16) -- the conditioning input of
// decoder_normalize's adaLN GEMMs, written here instead of by a separate conversion launch
__global__ void timestep_embed_kernel(const float* __restrict__ timestep, const int* __restrict__ step_ptr,
                                      const float* __restrict__ W, int B, int H, float* __restrict__ out, void* __restrict__ out16, int fmt16) {
  pdl_trigger();
  pdl_wait();  // predecessor grid complete + flushed before any dependent global access
  const int half = H / 2;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * half) return;
  const int b = i / half, j = i % half;
  const float t = step_ptr ? static_cast<float>(*step_ptr) : (timestep ? timestep[b] : static_cast<float>(b));
  // x[:, None] * W[None, :] * 2 * torch.pi  -> three separately rounded fp32 multiplies (model.py:95)
  const float x = __fmul_rn(__fmul_rn(__fmul_rn(t, W[j]), 2.0f), 3.14159274101257324f);
  const float sv = sinf(x), cv = cosf(x);
  out[static_cast<size_t>(b) * H + j] = sv;
  out[static_cast<size_t>(b) * H + half + j] = cv;
  if (out16) {
    if (fmt16 == 1) {
      bf16* o = static_cast<bf16*>(out16);
      o[static_cast<size_t>(b) * H + j] = from_f32<bf16>(sv);
      o[static_cast<size_t>(b) * H + half + j] = from_f32<bf16>(cv);
    } else {
      f16* o = static_cast<f16*>(out16);
      o[static_cast<size_t>(b) * H + j] = from_f32<f16>(sv);
      o[static_cast<size_t>(b) * H + half + j] = from_f32<f16>(cv);
    }
  }
}

int timestep_embed(const float* timestep, const int* step_ptr, const float* W, int B, int H, float* out, void* out16, int fmt16,
                   cudaStream_t s) {
  const int n = B * (H / 2);
  SD_CUDA(launch_k(timestep_embed_kernel, dim3(ceil_div(n, 128)), dim3(128), 0, s, timestep, step_ptr, W, B, H, out, out16, fmt16));
  SD_LAUNCHED("timestep_embed", s);
  return SEQDIFF_OK;
}

// ---------------------------------------------------------------------------------------------------
// BertEmbeddings (model.py:110-117), all embeddings of a forward in ONE launch.  A CTA serves one job (one embedding
// table): it stages that table's transposed weight [fin, H] in shared memory once -- before the PDL wait, weights do not
// depend on the predecessor -- and then walks the job's tokens, 4 tokens per warp pass so every weight vector read from
// smem is used 4x.  Input columns that are zero for all 4 tokens are skipped (adding 0 * w is exact): the one-hot sequence
// inputs touch at most 4 of their 20 weight rows.  (Before: every warp streamed the whole 61 KB table from L2 for its 4
// tokens, 250 MB per launch, 27 us x 4 launches per forward.)
template <typename T, int VPL>
__global__ void __launch_bounds__(kRowThreads, 2) embed_ln_multi_kernel(const __grid_constant__ EmbedJobs jobs, float eps, int H) {
  extern __shared__ float4 sW4[];
  float* sW = reinterpret_cast<float*>(sW4);
  int q = 0;
#pragma unroll
  for (int t = 1; t < 4; ++t)
    if (t < jobs.n && static_cast<int>(blockIdx.x) >= jobs.j[t].cta_begin) q = t;
  const EmbedJob& job = jobs.j[q];
  const int fin = job.fin, M = job.M;
  for (int i = threadIdx.x; i < fin * H / 4; i += kRowThreads) sW4[i] = __ldg(reinterpret_cast<const float4*>(job.Wt) + i);
  pdl_trigger();
  pdl_wait();  // inputs / timestep features come from the predecessor kernels
  if (jobs.cat_dst) {  // [mask_a | mask_b] for the stacked ligand|receptor attention (was two memcpy nodes per forward)
    for (int i = blockIdx.x * kRowThreads + threadIdx.x; i < jobs.cat_na + jobs.cat_nb; i += gridDim.x * kRowThreads)
      jobs.cat_dst[i] = i < jobs.cat_na ? __ldg(jobs.cat_a + i) : __ldg(jobs.cat_b + (i - jobs.cat_na));
  }
  __syncthreads();
  constexpr int TOK = kEmbedTok;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int cta_local = static_cast<int>(blockIdx.x) - job.cta_begin;
  T* outT = static_cast<T*>(job.outT);
  // the 4 x fin input values of a group are fetched with coalesced loads ONE GROUP AHEAD into a per-warp smem slot and read
  // back as broadcasts; scalar __ldg inside the k loop put a ~600-cycle global round trip on every k (66 us per launch)
  float* sx = sW + static_cast<size_t>(jobs.max_fin) * H + warp * (2 * TOK * 32);
  const int gstep = job.cta_count * (kRowThreads / 32);
  auto fetch_x = [&](int grp_n, int buf) {
    if (job.src_rows) {  // packed mode: output row r reads input row src_rows[r]
      for (int i = lane; i < TOK * fin; i += 32) {
        const int r = grp_n * TOK + i / fin;
        sx[buf * TOK * 32 + i] = r < M ? __ldg(job.x + static_cast<size_t>(__ldg(job.src_rows + r)) * fin + (i % fin)) : 0.f;
      }
      return;
    }
    const size_t base = static_cast<size_t>(grp_n) * TOK * fin;
    const size_t lim = static_cast<size_t>(M) * fin;
    for (int i = lane; i < TOK * fin; i += 32) sx[buf * TOK * 32 + i] = (base + i < lim) ? __ldg(job.x + base + i) : 0.f;
  };
  int xb = 0;
  {
    const int g0 = cta_local * (kRowThreads / 32) + warp;
    if (g0 * TOK < M) fetch_x(g0, 0);
    __syncwarp();
  }
  for (int grp = cta_local * (kRowThreads / 32) + warp; grp * TOK < M; grp += gstep, xb ^= 1) {
    const int tok0 = grp * TOK;
    if ((grp + gstep) * TOK < M) fetch_x(grp + gstep, xb ^ 1);  // next group's inputs: in flight during this group's math
    const float* xs = sx + xb * TOK * 32;
    float acc[TOK][VPL][8];
#pragma unroll
    for (int t = 0; t < TOK; ++t)
#pragma unroll
      for (int i = 0; i < VPL; ++i)
#pragma unroll
        for (int jj = 0; jj < 8; ++jj) acc[t][i][jj] = 0.f;
    for (int k = 0; k < fin; ++k) {
      float xv[TOK];
      bool any = false;
#pragma unroll
      for (int t = 0; t < TOK; ++t) {
        xv[t] = xs[t * fin + k];  // (rows past M were staged as zeros)
        any |= xv[t] != 0.f;
      }
      if (!any) continue;  // warp-uniform (every lane holds the same xv)
#pragma unroll
      for (int i = 0; i < VPL; ++i) {
        float w[8];
        load8<float>(sW + static_cast<size_t>(k) * H + (i * 32 + lane) * 8, w);
#pragma unroll
        for (int t = 0; t < TOK; ++t)
#pragma unroll
          for (int jj = 0; jj < 8; ++jj) acc[t][i][jj] = fmaf(xv[t], w[jj], acc[t][i][jj]);
      }
    }
#pragma unroll
    for (int t = 0; t < TOK; ++t) {
      if (tok0 + t >= M) break;
      float v[VPL][8];
#pragma unroll
      for (int i = 0; i < VPL; ++i) {
        float b8[8];
        load8<float>(job.b + (i * 32 + lane) * 8, b8);
#pragma unroll
        for (int jj = 0; jj < 8; ++jj) v[i][jj] = acc[t][i][jj] + b8[jj];
      }
      float mean, rstd;
      row_stats<VPL>(v, H, eps, mean, rstd);
      const int te_r = job.te_row ? *job.te_row : (job.row_graph ? __ldg(job.row_graph + tok0 + t) : (tok0 + t) / job.L);
      const float* terow = job.te ? job.te + static_cast<size_t>(te_r) * H : nullptr;
#pragma unroll
      for (int i = 0; i < VPL; ++i) {
        float g8[8], b8[8];
        load8<float>(job.lnw + (i * 32 + lane) * 8, g8);
        load8<float>(job.lnb + (i * 32 + lane) * 8, b8);
#pragma unroll
        for (int jj = 0; jj < 8; ++jj) v[i][jj] = (v[i][jj] - mean) * rstd * g8[jj] + b8[jj];
        if (terow) {
          float t8[8];
          load8<float>(terow + (i * 32 + lane) * 8, t8);
#pragma unroll
          for (int jj = 0; jj < 8; ++jj) v[i][jj] += t8[jj];
        }
      }
      if (job.out32) store_row<float, VPL>(job.out32 + static_cast<size_t>(tok0 + t) * H, lane, v);
      if (outT) store_row<T, VPL>(outT + static_cast<size_t>(tok0 + t) * H, lane, v);
    }
    __syncwarp();  // next group's staged inputs are complete; this group's slot may be overwritten in the next iteration
  }
}

#define SD_VPL_DISPATCH(H_, ...)                                        \
  switch ((H_) / 256) {                                                  \
    case 1: { constexpr int VPL = 1; __VA_ARGS__; } break;                      \
    case 2: { constexpr int VPL = 2; __VA_ARGS__; } break;                      \
    case 3: { constexpr int VPL = 3; __VA_ARGS__; } break;                      \
    case 4: { constexpr int VPL = 4; __VA_ARGS__; } break;                      \
    default: set_error("hidden_size must be 256, 512, 768 or 1024"); return SEQDIFF_ERR_INVALID; \
  }

template <typename T>
int embed_ln_multi(EmbedJobs jobs, float eps, int H, cudaStream_t s) {
  SD_CHECK(H % 256 == 0, "hidden_size must be a multiple of 256");
  SD_CHECK(jobs.n >= 1 && jobs.n <= 4, "1..4 embedding jobs per launch");
  // CTAs are shared out in proportion to the rows each job writes; one resident CTA per SM in total
  long total = 0;
  int max_fin = 0;
  for (int q = 0; q < jobs.n; ++q) {
    SD_CHECK(jobs.j[q].M > 0 && jobs.j[q].fin > 0 && jobs.j[q].fin <= 32 && jobs.j[q].L > 0, "bad embedding job");
    total += jobs.j[q].M;
    max_fin = jobs.j[q].fin > max_fin ? jobs.j[q].fin : max_fin;
  }
  const int budget = 2 * num_sms();  // two resident CTAs per SM
  int begin = 0;
  for (int q = 0; q < jobs.n; ++q) {
    int c = static_cast<int>(static_cast<long>(budget) * jobs.j[q].M / total);
    const int need = ceil_div(jobs.j[q].M, kEmbedTok * (kRowThreads / 32));
    if (c < 1) c = 1;
    if (c > need) c = need;
    jobs.j[q].cta_begin = begin;
    jobs.j[q].cta_count = c;
    begin += c;
  }
  jobs.max_fin = max_fin;
  const size_t smem = static_cast<size_t>(max_fin) * H * sizeof(float) + (kRowThreads / 32) * 2 * kEmbedTok * 32 * sizeof(float);
#define SD_EMBED_LAUNCH()                                                                                                          \
  {                                                                                                                                \
    auto kfn = embed_ln_multi_kernel<T, VPL>;                                                                                      \
    static bool configured = false;                                                                                                \
    if (!configured) {                                                                                                             \
      SD_CUDA(cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, 32 * 1024 * 4 + 8192));                       \
      configured = true;                                                                                                           \
    }                                                                                                                              \
    SD_CUDA(launch_k(kfn, dim3(begin), dim3(kRowThreads), smem, s, jobs, eps, H));                                                 \
  }
  SD_VPL_DISPATCH(H, SD_EMBED_LAUNCH());
#undef SD_EMBED_LAUNCH
  SD_LAUNCHED("embed_ln", s);
  return SEQDIFF_OK;
}
template int embed_ln_multi<float>(EmbedJobs, float, int, cudaStream_t);
template int embed_ln_multi<bf16>(EmbedJobs, float, int, cudaStream_t);
template int embed_ln_multi<f16>(EmbedJobs, float, int, cudaStream_t);

// ---------------------------------------------------------------------------------------------------
template <typename T, int VPL, int THREADS = kRowThreads, int RPW = 1>
__global__ void __launch_bounds__(THREADS) layernorm_kernel(const float* __restrict__ in, int M, int H, const float* __restrict__ w,
                                                            const float* __restrict__ b, float eps, float* __restrict__ out32,
                                                            T* __restrict__ outT, float2* __restrict__ stats) {
  pdl_trigger();
  pdl_wait();  // predecessor grid complete + flushed before any dependent global access
  const int lane = threadIdx.x & 31;
  const int row0 = ((blockIdx.x * THREADS + threadIdx.x) >> 5) * RPW;  // RPW consecutive rows per warp, all loads issued up front
  if (row0 >= M) return;
  float v[RPW][VPL][8];
#pragma unroll
  for (int r = 0; r < RPW; ++r)
    if (row0 + r < M) load_row<float, VPL>(in + static_cast<size_t>(row0 + r) * H, lane, v[r]);
#pragma unroll
  for (int r = 0; r < RPW; ++r) {
    const int row = row0 + r;
    if (row >= M) break;
    float mean, rstd;
    row_stats<VPL>(v[r], H, eps, mean, rstd);
    if (stats && lane == 0) stats[row] = make_float2(mean, rstd);  // lets a consumer re-derive LN(in) without the fp32 copy
#pragma unroll
    for (int i = 0; i < VPL; ++i) {
      float g8[8], b8[8];
      load8<float>(w + (i * 32 + lane) * 8, g8);
      load8<float>(b + (i * 32 + lane) * 8, b8);
#pragma unroll
      for (int j = 0; j < 8; ++j) v[r][i][j] = (v[r][i][j] - mean) * rstd * g8[j] + b8[j];
    }
    if (out32) store_row<float, VPL>(out32 + static_cast<size_t>(row) * H, lane, v[r]);
    if (outT) store_row<T, VPL>(outT + static_cast<size_t>(row) * H, lane, v[r]);
  }
}

template <typename T>
int layernorm(const float* in, int M, int H, const float* w, const float* b, float eps, float* out32, T* outT, float2* stats, cudaStream_t s) {
  // launch shape: SEQDIFF_LN_VAR = threads per CTA * 10 + rows per warp (sweep on B200: profiles/ln_sweep_r01.log)
  static const int var = [] { const char* e = getenv("SEQDIFF_LN_VAR"); return e ? atoi(e) : 2561; }();
#define SD_LN_LAUNCH(TH_, RPW_)                                                                                                           \
  {                                                                                                                                       \
    const int grid = ceil_div(ceil_div(M, RPW_) * 32, TH_);                                                                               \
    SD_VPL_DISPATCH(H, SD_CUDA(launch_k(layernorm_kernel<T, VPL, TH_, RPW_>, dim3(grid), dim3(TH_), 0, s, in, M, H, w, b, eps, out32, outT, stats))); \
  }
  switch (var) {
    case 1281: SD_LN_LAUNCH(128, 1); break;
    case 5121: SD_LN_LAUNCH(512, 1); break;
    case 2562: SD_LN_LAUNCH(256, 2); break;
    case 1282: SD_LN_LAUNCH(128, 2); break;
    case 641: SD_LN_LAUNCH(64, 1); break;
    default: SD_LN_LAUNCH(256, 1); break;
  }
#undef SD_LN_LAUNCH
  SD_LAUNCHED("layernorm", s);
  return SEQDIFF_OK;
}
#define SD_INST_LN(T) template int layernorm<T>(const float*, int, int, const float*, const float*, float, float*, T*, float2*, cudaStream_t)
SD_INST_LN(float);
SD_INST_LN(bf16);
SD_INST_LN(f16);

// ---------------------------------------------------------------------------------------------------
template <typename T, int VPL, bool AFFINE_FIRST>
__global__ void __launch_bounds__(kRowThreads) ln_modulate_kernel(const float* __restrict__ in, int M, int H, const float* __restrict__ lnw,
                                                                  const float* __restrict__ lnb, float eps1, const float* __restrict__ x,
                                                                  const T* __restrict__ mod, int mod_div, int chunk0,
                                                                  float* __restrict__ out32, T* __restrict__ outT, const int* __restrict__ row_graph,
                                                                  const int* __restrict__ mod_row, int split, const float* __restrict__ in_hi,
                                                                  const float* __restrict__ x_hi) {
  pdl_trigger();
  pdl_wait();  // predecessor grid complete + flushed before any dependent global access
  const int lane = threadIdx.x & 31;
  const int row = (blockIdx.x * kRowThreads + threadIdx.x) >> 5;
  if (row >= M) return;
  const bool hi = in_hi && row >= split;
  float v[VPL][8];
  load_row<float, VPL>(hi ? in_hi + static_cast<size_t>(row - split) * H : in + static_cast<size_t>(row) * H, lane, v);
  float mean, rstd;
  if (AFFINE_FIRST) {  // BertSelfOutput.LayerNorm (eps 1e-12, affine) -- output of self.attn(x, mask)[0]
    row_stats<VPL>(v, H, eps1, mean, rstd);
#pragma unroll
    for (int i = 0; i < VPL; ++i) {
      float g8[8], b8[8];
      load8<float>(lnw + (i * 32 + lane) * 8, g8);
      load8<float>(lnb + (i * 32 + lane) * 8, b8);
#pragma unroll
      for (int j = 0; j < 8; ++j) v[i][j] = (v[i][j] - mean) * rstd * g8[j] + b8[j];
    }
  }
  row_stats<VPL>(v, H, 1e-5f, mean, rstd);  // SELayer.norm1/norm2: elementwise_affine=False, default eps
  SD_DEV_ASSERT(!row_graph || __ldg(row_graph + row) >= 0);
  SD_DEV_ASSERT(!mod_row || *mod_row >= 0);
  const int mr = mod_row ? *mod_row : (row_graph ? __ldg(row_graph + row) : row / mod_div);
  const T* mrow = mod + static_cast<size_t>(mr) * (6 * H);
  const float* xrow = hi ? x_hi + static_cast<size_t>(row - split) * H : x + static_cast<size_t>(row) * H;
#pragma unroll
  for (int i = 0; i < VPL; ++i) {
    const int e = (i * 32 + lane) * 8;
    float sh[8], sc[8], gt[8], xr[8];
    load8<T>(mrow + (chunk0 + 0) * H + e, sh);
    load8<T>(mrow + (chunk0 + 1) * H + e, sc);
    load8<T>(mrow + (chunk0 + 2) * H + e, gt);
    load8<float>(xrow + e, xr);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float n = (v[i][j] - mean) * rstd;
      v[i][j] = xr[j] + gt[j] * (n * (1.0f + sc[j]) + sh[j]);
    }
  }
  if (out32) store_row<float, VPL>(out32 + static_cast<size_t>(row) * H, lane, v);
  if (outT) store_row<T, VPL>(outT + static_cast<size_t>(row) * H, lane, v);
}

template <typename T>
int ln_modulate(const float* in, int M, int H, bool affine_first, const float* lnw, const float* lnb, float eps1, const float* x,
                const T* mod, int mod_div, int chunk0, float* out32, T* outT, cudaStream_t s, const int* row_graph, const int* mod_row, int split,
                const float* in_hi, const float* x_hi) {
  SD_CHECK(!in_hi == !x_hi && (!in_hi || (split >= 0 && split <= M)), "ln_modulate: split sources need both in_hi and x_hi and 0 <= split <= M");
  const int grid = ceil_div(M * 32, kRowThreads);
  if (affine_first) {
    SD_VPL_DISPATCH(H, SD_CUDA(launch_k(ln_modulate_kernel<T, VPL, true>, dim3(grid), dim3(kRowThreads), 0, s, in, M, H, lnw, lnb, eps1, x, mod, mod_div, chunk0, out32, outT, row_graph,
                                        mod_row, split, in_hi, x_hi)));
  } else {
    SD_VPL_DISPATCH(H, SD_CUDA(launch_k(ln_modulate_kernel<T, VPL, false>, dim3(grid), dim3(kRowThreads), 0, s, in, M, H, lnw, lnb, eps1, x, mod, mod_div, chunk0, out32, outT, row_graph,
                                        mod_row, split, in_hi, x_hi)));
  }
  SD_LAUNCHED("ln_modulate", s);
  return SEQDIFF_OK;
}
#define SD_INST_LNMOD(T)                                                                                                                                  \
  template int ln_modulate<T>(const float*, int, int, bool, const float*, const float*, float, const float*, const T*, int, int, float*, T*, cudaStream_t, \
                              const int*, const int*, int, const float*, const float*)
SD_INST_LNMOD(float);
SD_INST_LNMOD(bf16);
SD_INST_LNMOD(f16);

// ---------------------------------------------------------------------------------------------------
// W2 [F, H] is staged in shared memory once per CTA (before the PDL wait) and every CTA walks its share of the rows, 4 rows
// per warp pass so each weight vector read from smem serves 4 rows.  (Before: one row per warp, each warp streaming all of
// W2 -- 61 KB -- from L2: 500 MB and 54 us per launch for 126 MFLOP.)
template <typename T, int VPL>
__global__ void __launch_bounds__(kRowThreads) predictor_tail_kernel(const T* __restrict__ y, int M, int H, const float* __restrict__ lnw,
                                                                     const float* __restrict__ lnb, float eps,
                                                                     const float* __restrict__ W2, const float* __restrict__ b2, int F,
                                                                     float* __restrict__ logits, const int* __restrict__ dst_rows) {
  extern __shared__ float4 sW4[];
  float* sW = reinterpret_cast<float*>(sW4);
  for (int i = threadIdx.x; i < F * H / 4; i += kRowThreads) sW4[i] = __ldg(reinterpret_cast<const float4*>(W2) + i);
  float* sG = sW + static_cast<size_t>(F) * H;  // LayerNorm weight | bias
  for (int i = threadIdx.x; i < H; i += kRowThreads) {
    sG[i] = __ldg(lnw + i);
    sG[H + i] = __ldg(lnb + i);
  }
  pdl_trigger();
  pdl_wait();  // predecessor grid complete + flushed before any dependent global access
  __syncthreads();
  constexpr int ROWS = 4;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const float bias_f = lane < F ? b2[lane] : 0.f;
  for (int grp = blockIdx.x * (kRowThreads / 32) + warp; grp * ROWS < M; grp += gridDim.x * (kRowThreads / 32)) {
    const int row0 = grp * ROWS;
    float v[ROWS][VPL][8];
#pragma unroll
    for (int r = 0; r < ROWS; ++r) {
      const int row = row0 + r < M ? row0 + r : M - 1;  // tail rows recompute the last row (not stored)
      load_row<T, VPL>(y + static_cast<size_t>(row) * H, lane, v[r]);
      float mean, rstd;
      row_stats<VPL>(v[r], H, eps, mean, rstd);
#pragma unroll
      for (int i = 0; i < VPL; ++i) {
        float g8[8], be8[8];
        load8<float>(sG + (i * 32 + lane) * 8, g8);
        load8<float>(sG + H + (i * 32 + lane) * 8, be8);
#pragma unroll
        for (int jj = 0; jj < 8; ++jj) v[r][i][jj] = (v[r][i][jj] - mean) * rstd * g8[jj] + be8[jj];
      }
    }
    float mine[ROWS];  // lane f keeps logit f of each row
#pragma unroll
    for (int r = 0; r < ROWS; ++r) mine[r] = 0.f;
    for (int f = 0; f < F; ++f) {
      float p[ROWS];
#pragma unroll
      for (int r = 0; r < ROWS; ++r) p[r] = 0.f;
#pragma unroll
      for (int i = 0; i < VPL; ++i) {
        float w[8];
        load8<float>(sW + static_cast<size_t>(f) * H + (i * 32 + lane) * 8, w);
#pragma unroll
        for (int r = 0; r < ROWS; ++r)
#pragma unroll
          for (int jj = 0; jj < 8; ++jj) p[r] = fmaf(v[r][i][jj], w[jj], p[r]);
      }
#pragma unroll
      for (int r = 0; r < ROWS; ++r) {
        p[r] = warp_sum(p[r]);
        if (lane == f) mine[r] = p[r] + bias_f;
      }
    }
#pragma unroll
    for (int r = 0; r < ROWS; ++r)
      if (lane < F && row0 + r < M) logits[static_cast<size_t>(dst_rows ? __ldg(dst_rows + row0 + r) : row0 + r) * F + lane] = mine[r];
  }
}

template <typename T>
int predictor_tail(const T* y, int M, int H, const float* lnw, const float* lnb, float eps, const float* W2, const float* b2, int F,
                   float* logits, cudaStream_t s, const int* dst_rows) {
  SD_CHECK(F <= 32, "feature_size > 32 not supported");
  const int need = ceil_div(M, 4 * (kRowThreads / 32));
  const int grid = need < num_sms() ? need : num_sms();  // ~185 registers x 256 threads: one CTA per SM
  const size_t smem = (static_cast<size_t>(F) + 2) * H * sizeof(float);
#define SD_PRED_LAUNCH()                                                                                              \
  {                                                                                                                   \
    auto kfn = predictor_tail_kernel<T, VPL>;                                                                         \
    static bool configured = false;                                                                                   \
    if (!configured) {                                                                                                \
      SD_CUDA(cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, 34 * 1024 * 4));                 \
      configured = true;                                                                                              \
    }                                                                                                                 \
    SD_CUDA(launch_k(kfn, dim3(grid), dim3(kRowThreads), smem, s, y, M, H, lnw, lnb, eps, W2, b2, F, logits, dst_rows)); \
  }
  SD_VPL_DISPATCH(H, SD_PRED_LAUNCH());
#undef SD_PRED_LAUNCH
  SD_LAUNCHED("predictor_tail", s);
  return SEQDIFF_OK;
}
template int predictor_tail<float>(const float*, int, int, const float*, const float*, float, const float*, const float*, int, float*, cudaStream_t, const int*);
template int predictor_tail<bf16>(const bf16*, int, int, const float*, const float*, float, const float*, const float*, int, float*, cudaStream_t, const int*);
template int predictor_tail<f16>(const f16*, int, int, const float*, const float*, float, const float*, const float*, int, float*, cudaStream_t, const int*);

// ---------------------------------------------------------------------------------------------------
template <typename T>
__global__ void f32_to_16_kernel(const float* __restrict__ in, size_t n, T* __restrict__ out) {
  pdl_trigger();
  pdl_wait();  // predecessor grid complete + flushed before any dependent global access
  size_t i = (static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x);
  const size_t stride = static_cast<size_t>(gridDim.x) * blockDim.x;
  const size_t n4 = ((reinterpret_cast<uintptr_t>(in) & 15) == 0 && (reinterpret_cast<uintptr_t>(out) & 7) == 0) ? n / 4 : 0;
  for (size_t v = i; v < n4; v += stride) {  // 16 B in, 8 B out per thread
    const float4 a = *reinterpret_cast<const float4*>(in + 4 * v);
    *reinterpret_cast<uint2*>(out + 4 * v) = make_uint2(pack2<T>(a.x, a.y), pack2<T>(a.z, a.w));
  }
  for (i += 4 * n4; i < n; i += stride) out[i] = from_f32<T>(in[i]);
}
template <typename T>
int f32_to_16(const float* in, size_t n, T* out, cudaStream_t s) {
  if (n == 0) return SEQDIFF_OK;
  size_t blocks = (n + 255) / 256;
  if (blocks > 4096) blocks = 4096;
  SD_CUDA(launch_k(f32_to_16_kernel<T>, dim3(static_cast<int>(blocks)), dim3(256), 0, s, in, n, out));
  SD_LAUNCHED("f32_to_16", s);
  return SEQDIFF_OK;
}
template int f32_to_16<bf16>(const float*, size_t, bf16*, cudaStream_t);
template int f32_to_16<f16>(const float*, size_t, f16*, cudaStream_t);

__global__ void transpose_f32_kernel(const float* __restrict__ in, int rows, int cols, float* __restrict__ out) {
  pdl_trigger();
  pdl_wait();  // predecessor grid complete + flushed before any dependent global access
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * cols) return;
  const int r = i / cols, c = i % cols;
  out[static_cast<size_t>(c) * rows + r] = in[i];
}
int transpose_f32(const float* in, int rows, int cols, float* out, cudaStream_t s) {
  SD_CUDA(launch_k(transpose_f32_kernel, dim3(ceil_div(rows * cols, 256)), dim3(256), 0, s, in, rows, cols, out));
  SD_LAUNCHED("transpose_f32", s);
  return SEQDIFF_OK;
}

__global__ void step_advance_kernel(int* p) {
  pdl_trigger();
  pdl_wait();
  *p -= 1;
}
int step_advance(int* step_ptr, cudaStream_t s) {
  SD_CUDA(launch_k(step_advance_kernel, dim3(1), dim3(1), 0, s, step_ptr));
  SD_LAUNCHED("step_advance", s);
  return SEQDIFF_OK;
}

}  // namespace seqdiff
