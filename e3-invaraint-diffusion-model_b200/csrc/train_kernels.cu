// train_kernels.cu -- the rowwise / elementwise kernels of the TRAINING step (BASELINE configs[3]; reference
// sequence_model/model.py:313-367 `get_loss` + `training_step` under autograd, train_model.py:30-33,95 AdamW + clip):
// dropout, activation forward / backward, LayerNorm and adaLN-modulate backward, embedding / predictor-tail backward, the loss
// gradient, 16-bit transposes for the weight-gradient GEMMs, and the fused clip + AdamW update.
//
// Conventions.  Gradients of the residual stream are fp32 [rows, H]; gradients that feed a tensor-core GEMM are also written
// in the operand type T (bf16 / fp16; fp32 in the parity mode).  One warp owns one token row (H = 256 * VPL).  Parameter
// gradients that are sums over rows (biases, LayerNorm affine, embedding / predictor weights) are reduced per CTA in shared
// memory and flushed with one atomicAdd per element and CTA into the flat fp32 gradient buffer, which the step zeroes first.
// Dropout masks are never stored: forward and backward regenerate them from Philox4x32-10 keyed by (seed, site, element).
#include <cstdlib>

#include "common.cuh"
#include "kernels.h"
#include "philox.cuh"

namespace seqdiff {

constexpr int kTrThreads = 256;

template <typename T, int VPL>
__device__ __forceinline__ void ld_row(const T* __restrict__ row, int lane, float (&v)[VPL][8]) {
#pragma unroll
  for (int i = 0; i < VPL; ++i) load8<T>(row + (i * 32 + lane) * 8, v[i]);
}
template <typename T, int VPL>
__device__ __forceinline__ void st_row(T* __restrict__ row, int lane, const float (&v)[VPL][8]) {
#pragma unroll
  for (int i = 0; i < VPL; ++i) store8<T>(row + (i * 32 + lane) * 8, v[i]);
}
// (mean, rstd) exactly as the forward kernels compute them (rowwise.cu: row_stats)
template <int VPL>
__device__ __forceinline__ void stats_of(const float (&v)[VPL][8], int H, float eps, float& mean, float& rstd) {
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
  rstd = 1.0f / sqrtf(warp_sum(q) / static_cast<float>(H) + eps);
}
// y = (x - mean) * rstd (no affine).  In: xhat (normalised values), g = dL/dy.  Out (in g): dL/dx = rstd * (g - mean(g) - xhat * mean(g * xhat))
template <int VPL>
__device__ __forceinline__ void ln_bwd_core(const float (&xhat)[VPL][8], float (&g)[VPL][8], int H, float rstd) {
  float s1 = 0.f, s2 = 0.f;
#pragma unroll
  for (int i = 0; i < VPL; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      s1 += g[i][j];
      s2 = fmaf(g[i][j], xhat[i][j], s2);
    }
  s1 = warp_sum(s1) / static_cast<float>(H);
  s2 = warp_sum(s2) / static_cast<float>(H);
#pragma unroll
  for (int i = 0; i < VPL; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) g[i][j] = rstd * (g[i][j] - s1 - xhat[i][j] * s2);
}

#define SD_VPL_DISPATCH(H_, ...)                                        \
  switch ((H_) / 256) {                                                  \
    case 1: { constexpr int VPL = 1; __VA_ARGS__; } break;                      \
    case 2: { constexpr int VPL = 2; __VA_ARGS__; } break;                      \
    case 3: { constexpr int VPL = 3; __VA_ARGS__; } break;                      \
    case 4: { constexpr int VPL = 4; __VA_ARGS__; } break;                      \
    default: set_error("hidden_size must be 256, 512, 768 or 1024"); return SEQDIFF_ERR_INVALID; \
  }

// =====================================================================================================
// transposes: out[c][r] = in[r][c] for a row-major [rows, cols] matrix of T; optional column sums (bias gradients)
// =====================================================================================================
template <typename T>
__global__ void __launch_bounds__(256) transpose_colsum_kernel(const T* __restrict__ in, int rows, int cols, T* __restrict__ out, int pitch,
                                                               float* __restrict__ colsum) {
  pdl_wait();
  __shared__ float tile[64][65];
  const int r0 = blockIdx.y * 64, c0 = blockIdx.x * 64;
  const int tx = threadIdx.x & 63, ty = threadIdx.x >> 6;  // 64 x 4
  float cs = 0.f;
#pragma unroll 4
  for (int i = ty; i < 64; i += 4) {
    const int r = r0 + i, c = c0 + tx;
    const float v = (r < rows && c < cols) ? to_f32<T>(in[static_cast<size_t>(r) * cols + c]) : 0.f;
    tile[i][tx] = v;
    cs += v;
  }
  if (colsum) {  // 4 partial sums per column -> smem -> one atomic per column and CTA
    __shared__ float part[4][64];
    part[ty][tx] = cs;
    __syncthreads();
    if (ty == 0 && c0 + tx < cols) atomicAdd(colsum + c0 + tx, part[0][tx] + part[1][tx] + part[2][tx] + part[3][tx]);
  } else {
    __syncthreads();
  }
  if (out) {
#pragma unroll 4
    for (int i = ty; i < 64; i += 4) {
      const int c = c0 + i, r = r0 + tx;
      if (c < cols && r < pitch) out[static_cast<size_t>(c) * pitch + r] = from_f32<T>(tile[tx][i]);  // rows..pitch-1: zero padding
    }
  }
}
template <typename T>
int transpose_colsum(const T* in, int rows, int cols, T* out, float* colsum, cudaStream_t s, int pitch) {
  SD_CHECK(rows > 0 && cols > 0, "empty transpose");
  if (pitch <= 0) pitch = rows;
  SD_CHECK(pitch >= rows && pitch - rows < 64, "transpose: pitch must be rows rounded up by less than one tile");
  SD_CUDA(launch_k(transpose_colsum_kernel<T>, dim3(ceil_div(cols, 64), ceil_div(pitch, 64)), dim3(256), 0, s, in, rows, cols, out, pitch, colsum));
  SD_LAUNCHED("transpose", s);
  return SEQDIFF_OK;
}
template int transpose_colsum<float>(const float*, int, int, float*, float*, cudaStream_t, int);
template int transpose_colsum<bf16>(const bf16*, int, int, bf16*, float*, cudaStream_t, int);
template int transpose_colsum<f16>(const f16*, int, int, f16*, float*, cudaStream_t, int);

// Shared-memory accumulators that every row of a warp adds into: column e = (i * 32 + lane) * 8 + j of a feature row lives in slot
// (i * 8 + j) * 32 + lane, so the 32 lanes of one atomic instruction hit 32 different banks (with the natural index they are 8 words
// apart: 8-way conflicts on every one of the ~10 k shared atomics per row -- ncu: embed_bwd 274 us per launch).
__device__ __forceinline__ int acc_slot(int i, int lane, int j) { return (i * 8 + j) * 32 + lane; }
__device__ __forceinline__ int acc_slot_of_col(int e) { return acc_slot(e >> 8, (e >> 3) & 31, e & 7); }
// End-of-kernel flush of per-CTA partial sums into the flat gradient buffer.  Every CTA of the grid adds to the SAME few thousand addresses
// at the same moment, and same-address atomics serialise in L2 (ncu launch list of a training step: embed_bwd 80 - 113 us per launch, almost
// all of it the 6 - 15 k scalar atomics per CTA): four consecutive elements go as ONE 128-bit atomic (sm_90+: atomicAdd(float4*)) whenever
// the destination is 16 B aligned -- a quarter of the operations on the contended addresses.
__device__ __forceinline__ bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }
__device__ __forceinline__ void atomic_add4(float* dst, float a, float b, float c, float d) {
  atomicAdd(reinterpret_cast<float4*>(dst), make_float4(a, b, c, d));
}

// column sums of a 16-bit / fp32 [rows, cols] matrix, ADDED into colsum[cols] (pre-zeroed): the bias gradient db = sum over tokens of dY
// when the weight-gradient GEMM reads dY in place (gemm_16_tn) and no transpose pass exists to fuse it into.
// Block = 32 column-octets x 8 row lanes over a slab of 64 rows (enough CTAs to fill the GPU at M = 2048 .. 32768 rows); partial sums
// meet in shared memory, one atomic per column and CTA.
template <typename T>
__global__ void __launch_bounds__(256) colsum_kernel(const T* __restrict__ in, int rows, int cols, float* __restrict__ colsum) {
  pdl_wait();
  __shared__ float part[8][256];
  const int oct = threadIdx.x & 31, rl = threadIdx.x >> 5;
  const int c0 = blockIdx.x * 256 + oct * 8;
  const int r0 = blockIdx.y * 64;
  float acc[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) acc[j] = 0.f;
  if (c0 < cols) {
    const int r_end = r0 + 64 < rows ? r0 + 64 : rows;
    for (int r = r0 + rl; r < r_end; r += 8) {
      float x[8];
      load8<T>(in + static_cast<size_t>(r) * cols + c0, x);
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[j] += x[j];
    }
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) part[rl][oct * 8 + j] = acc[j];
  __syncthreads();
  // rows / 64 CTAs add to the same `cols` addresses: four columns per 128-bit atomic when the destination allows it (cols % 8 == 0)
  if (aligned16(colsum)) {
    const int c = blockIdx.x * 256 + 4 * threadIdx.x;
    if (threadIdx.x < 64 && c < cols) {
      float sum[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int u = 0; u < 4; ++u) sum[u] += part[i][4 * threadIdx.x + u];
      atomic_add4(colsum + c, sum[0], sum[1], sum[2], sum[3]);
    }
  } else {
    const int c = blockIdx.x * 256 + threadIdx.x;
    if (c < cols) {
      float sum = 0.f;
#pragma unroll
      for (int i = 0; i < 8; ++i) sum += part[i][threadIdx.x];
      atomicAdd(colsum + c, sum);
    }
  }
}
template <typename T>
int colsum_add(const T* in, int rows, int cols, float* colsum, cudaStream_t s) {
  SD_CHECK(rows > 0 && cols > 0 && cols % 8 == 0, "colsum: cols must be a multiple of 8");
  SD_CUDA(launch_k(colsum_kernel<T>, dim3(ceil_div(cols, 256), ceil_div(rows, 64)), dim3(256), 0, s, in, rows, cols, colsum));
  SD_LAUNCHED("colsum", s);
  return SEQDIFF_OK;
}
template int colsum_add<bf16>(const bf16*, int, int, float*, cudaStream_t);
template int colsum_add<f16>(const f16*, int, int, float*, cudaStream_t);

// fp32 [rows, cols] -> T [cols, rows] (weights: the fp32 master -> the transposed operand copy the dgrad GEMMs read)
template <typename T>
__global__ void __launch_bounds__(256) transpose_cast_kernel(const float* __restrict__ in, int rows, int cols, T* __restrict__ out) {
  pdl_wait();
  __shared__ float tile[64][65];
  const int r0 = blockIdx.y * 64, c0 = blockIdx.x * 64;
  const int tx = threadIdx.x & 63, ty = threadIdx.x >> 6;
#pragma unroll 4
  for (int i = ty; i < 64; i += 4) {
    const int r = r0 + i, c = c0 + tx;
    tile[i][tx] = (r < rows && c < cols) ? in[static_cast<size_t>(r) * cols + c] : 0.f;
  }
  __syncthreads();
#pragma unroll 4
  for (int i = ty; i < 64; i += 4) {
    const int c = c0 + i, r = r0 + tx;
    if (c < cols && r < rows) out[static_cast<size_t>(c) * rows + r] = from_f32<T>(tile[tx][i]);
  }
}
template <typename T>
int transpose_cast(const float* in, int rows, int cols, T* out, cudaStream_t s) {
  SD_CUDA(launch_k(transpose_cast_kernel<T>, dim3(ceil_div(cols, 64), ceil_div(rows, 64)), dim3(256), 0, s, in, rows, cols, out));
  SD_LAUNCHED("transpose_w", s);
  return SEQDIFF_OK;
}
template int transpose_cast<float>(const float*, int, int, float*, cudaStream_t);
template int transpose_cast<bf16>(const float*, int, int, bf16*, cudaStream_t);
template int transpose_cast<f16>(const float*, int, int, f16*, cudaStream_t);

// =====================================================================================================
// activations and dropout
// =====================================================================================================
__device__ __forceinline__ float gelu_grad(float x) {  // d/dx [0.5 x (1 + erf(x / sqrt 2))]
  const float cdf = 0.5f * (1.0f + erff(x * 0.70710678118654752440f));
  return cdf + x * 0.3989422804014327f * expf(-0.5f * x * x);
}
__device__ __forceinline__ float silu_grad(float x) {
  const float sg = 1.0f / (1.0f + expf(-x));
  return sg * (1.0f + x * (1.0f - sg));
}

// a = dropout(act(z)); kind 1 = erf-GELU, 2 = SiLU.  8 elements per thread.
template <typename T>
__global__ void __launch_bounds__(256) act_fwd_kernel(const T* __restrict__ z, size_t n8, int kind, DropSpec dr, T* __restrict__ a) {
  pdl_wait();
  for (size_t i = static_cast<size_t>(blockIdx.x) * 256 + threadIdx.x; i < n8; i += static_cast<size_t>(gridDim.x) * 256) {
    float v[8];
    load8<T>(z + 8 * i, v);
    float keep[8];
    drop_scales8(dr, 8 * i, keep);
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = (kind == 1 ? gelu_erf(v[j]) : silu(v[j])) * keep[j];
    store8<T>(a + 8 * i, v);
  }
}
template <typename T>
int act_fwd(const T* z, size_t n, int kind, DropSpec dr, T* a, cudaStream_t s) {
  SD_CHECK(n % 8 == 0 && (kind == 1 || kind == 2), "act_fwd: n % 8 and kind");
  const size_t n8 = n / 8;
  const int grid = static_cast<int>(n8 / 256 + 1 < 2048 ? n8 / 256 + 1 : 2048);
  SD_CUDA(launch_k(act_fwd_kernel<T>, dim3(grid), dim3(256), 0, s, z, n8, kind, dr, a));
  SD_LAUNCHED("act_fwd", s);
  return SEQDIFF_OK;
}
// dz = da * keep * act'(z).  TG = type of the incoming gradient (T from a GEMM, float from a rowwise kernel).
template <typename T, typename TG>
__global__ void __launch_bounds__(256) act_bwd_kernel(const TG* __restrict__ da, const T* __restrict__ z, size_t n8, int kind, DropSpec dr,
                                                      T* __restrict__ dz) {
  pdl_wait();
  for (size_t i = static_cast<size_t>(blockIdx.x) * 256 + threadIdx.x; i < n8; i += static_cast<size_t>(gridDim.x) * 256) {
    float g[8], v[8], keep[8];
    load8<TG>(da + 8 * i, g);
    load8<T>(z + 8 * i, v);
    drop_scales8(dr, 8 * i, keep);
#pragma unroll
    for (int j = 0; j < 8; ++j) g[j] = g[j] * keep[j] * (kind == 1 ? gelu_grad(v[j]) : silu_grad(v[j]));
    store8<T>(dz + 8 * i, g);
  }
}
template <typename T, typename TG>
int act_bwd(const TG* da, const T* z, size_t n, int kind, DropSpec dr, T* dz, cudaStream_t s) {
  SD_CHECK(n % 8 == 0 && (kind == 1 || kind == 2), "act_bwd: n % 8 and kind");
  const size_t n8 = n / 8;
  const int grid = static_cast<int>(n8 / 256 + 1 < 2048 ? n8 / 256 + 1 : 2048);
  SD_CUDA(launch_k(act_bwd_kernel<T, TG>, dim3(grid), dim3(256), 0, s, da, z, n8, kind, dr, dz));
  SD_LAUNCHED("act_bwd", s);
  return SEQDIFF_OK;
}
// o = dropout(d) + resid (fp32, in place on d): the hidden-state dropout that sits between a Linear and its residual add
__global__ void __launch_bounds__(256) dropout_add_kernel(float* __restrict__ d, const float* __restrict__ resid, size_t n8, DropSpec dr) {
  pdl_wait();
  for (size_t i = static_cast<size_t>(blockIdx.x) * 256 + threadIdx.x; i < n8; i += static_cast<size_t>(gridDim.x) * 256) {
    float v[8], r[8], keep[8];
    load8<float>(d + 8 * i, v);
    drop_scales8(dr, 8 * i, keep);
    if (resid) {
      load8<float>(resid + 8 * i, r);
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = fmaf(v[j], keep[j], r[j]);
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] *= keep[j];
    }
    store8<float>(d + 8 * i, v);
  }
}
int dropout_add(float* d, const float* resid, size_t n, DropSpec dr, cudaStream_t s) {
  SD_CHECK(n % 8 == 0, "dropout_add: n % 8");
  const size_t n8 = n / 8;
  const int grid = static_cast<int>(n8 / 256 + 1 < 2048 ? n8 / 256 + 1 : 2048);
  SD_CUDA(launch_k(dropout_add_kernel, dim3(grid), dim3(256), 0, s, d, resid, n8, dr));
  SD_LAUNCHED("dropout_add", s);
  return SEQDIFF_OK;
}
// o = dropout(d) + resid (in place on d) AND h = LayerNorm(o) * w + b in one pass: the post-LN sublayers of the decoder
// (BertSelfOutput / BertOutput: dense -> dropout -> + residual -> LayerNorm).  o stays in memory for the backward pass; compared with
// dropout_add + layernorm the row is read and written once less (100 MB per launch at 16384 x 768) and one launch disappears.
// keep_bits (optional): the mask of the row as bits -- byte [row][i][lane] holds the 8 keep flags of elements (i * 32 + lane) * 8 .. + 7 --
// so that the LayerNorm backward of this sublayer does not have to regenerate it from Philox (half of its instruction stream).
template <typename T, int VPL>
__global__ void __launch_bounds__(kTrThreads) dropout_add_layernorm_kernel(float* __restrict__ d, const float* __restrict__ resid, DropSpec dr, int M,
                                                                           int H, const float* __restrict__ w, const float* __restrict__ b, float eps,
                                                                           float* __restrict__ out32, T* __restrict__ outT,
                                                                           uint8_t* __restrict__ keep_bits) {
  pdl_wait();
  const int lane = threadIdx.x & 31;
  const int row = (blockIdx.x * kTrThreads + threadIdx.x) >> 5;
  if (row >= M) return;
  float v[VPL][8], r[VPL][8];
  ld_row<float, VPL>(d + static_cast<size_t>(row) * H, lane, v);
  ld_row<float, VPL>(resid + static_cast<size_t>(row) * H, lane, r);
#pragma unroll
  for (int i = 0; i < VPL; ++i) {
    float keep[8];
    drop_scales8(dr, static_cast<size_t>(row) * H + (i * 32 + lane) * 8, keep);
    uint32_t bits = 0;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      v[i][j] = fmaf(v[i][j], keep[j], r[i][j]);
      bits |= (keep[j] != 0.f ? 1u : 0u) << j;
    }
    if (keep_bits) keep_bits[static_cast<size_t>(row) * (H / 8) + i * 32 + lane] = static_cast<uint8_t>(bits);
  }
  st_row<float, VPL>(d + static_cast<size_t>(row) * H, lane, v);
  float mean, rstd;
  stats_of<VPL>(v, H, eps, mean, rstd);
#pragma unroll
  for (int i = 0; i < VPL; ++i) {
    float g8[8], b8[8];
    load8<float>(w + (i * 32 + lane) * 8, g8);
    load8<float>(b + (i * 32 + lane) * 8, b8);
#pragma unroll
    for (int j = 0; j < 8; ++j) v[i][j] = (v[i][j] - mean) * rstd * g8[j] + b8[j];
  }
  if (out32) st_row<float, VPL>(out32 + static_cast<size_t>(row) * H, lane, v);
  if (outT) st_row<T, VPL>(outT + static_cast<size_t>(row) * H, lane, v);
}
template <typename T>
int dropout_add_layernorm(float* d, const float* resid, DropSpec dr, int M, int H, const float* w, const float* b, float eps, float* out32, T* outT,
                          uint8_t* keep_bits, cudaStream_t s) {
  SD_CHECK(M > 0 && resid, "dropout_add_layernorm: empty input");
  SD_VPL_DISPATCH(H, SD_CUDA(launch_k(dropout_add_layernorm_kernel<T, VPL>, dim3(ceil_div(M, kTrThreads / 32)), dim3(kTrThreads), 0, s, d, resid, dr, M,
                                      H, w, b, eps, out32, outT, keep_bits)));
  SD_LAUNCHED("dropout_add_ln", s);
  return SEQDIFF_OK;
}
template int dropout_add_layernorm<float>(float*, const float*, DropSpec, int, int, const float*, const float*, float, float*, float*, uint8_t*,
                                          cudaStream_t);
template int dropout_add_layernorm<bf16>(float*, const float*, DropSpec, int, int, const float*, const float*, float, float*, bf16*, uint8_t*,
                                         cudaStream_t);
template int dropout_add_layernorm<f16>(float*, const float*, DropSpec, int, int, const float*, const float*, float, float*, f16*, uint8_t*,
                                        cudaStream_t);
// gT = T(g * keep): the fp32 gradient of a (dropout-ed) Linear output as the 16-bit operand of its backward GEMMs
template <typename T>
__global__ void __launch_bounds__(256) grad_cast_kernel(const float* __restrict__ g, size_t n8, DropSpec dr, T* __restrict__ out) {
  pdl_wait();
  for (size_t i = static_cast<size_t>(blockIdx.x) * 256 + threadIdx.x; i < n8; i += static_cast<size_t>(gridDim.x) * 256) {
    float v[8], keep[8];
    load8<float>(g + 8 * i, v);
    drop_scales8(dr, 8 * i, keep);
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] *= keep[j];
    store8<T>(out + 8 * i, v);
  }
}
template <typename T>
int grad_cast(const float* g, size_t n, DropSpec dr, T* out, cudaStream_t s) {
  SD_CHECK(n % 8 == 0, "grad_cast: n % 8");
  const size_t n8 = n / 8;
  const int grid = static_cast<int>(n8 / 256 + 1 < 2048 ? n8 / 256 + 1 : 2048);
  SD_CUDA(launch_k(grad_cast_kernel<T>, dim3(grid), dim3(256), 0, s, g, n8, dr, out));
  SD_LAUNCHED("grad_cast", s);
  return SEQDIFF_OK;
}
#define SD_INST_ACT(T)                                                                              \
  template int act_fwd<T>(const T*, size_t, int, DropSpec, T*, cudaStream_t);                       \
  template int act_bwd<T, T>(const T*, const T*, size_t, int, DropSpec, T*, cudaStream_t);          \
  template int grad_cast<T>(const float*, size_t, DropSpec, T*, cudaStream_t)
SD_INST_ACT(float);
SD_INST_ACT(bf16);
SD_INST_ACT(f16);
template int act_bwd<bf16, float>(const float*, const bf16*, size_t, int, DropSpec, bf16*, cudaStream_t);
template int act_bwd<f16, float>(const float*, const f16*, size_t, int, DropSpec, f16*, cudaStream_t);

// =====================================================================================================
// LayerNorm backward (affine): h = LN(o) * g + b.  dh [M,H] fp32 -> do [M,H] fp32, dg / db accumulated
// =====================================================================================================
// CTA-level accumulation of per-feature sums: every warp adds its rows into registers, the warps of a CTA meet in smem, one
// atomicAdd per feature and CTA.  Grid-stride over rows so that the number of atomics stays ~ #CTAs * H.
template <int VPL>
__device__ __forceinline__ void flush_feature_sums(float (&acc)[VPL][8], float* __restrict__ dst, float* smem_acc /*[H]*/, int H, int lane) {
  // caller has zeroed smem_acc and synchronised; conflict-free slots (acc_slot), four columns per global atomic
#pragma unroll
  for (int i = 0; i < VPL; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) atomicAdd(smem_acc + acc_slot(i, lane, j), acc[i][j]);
  __syncthreads();
  if (aligned16(dst)) {
    for (int e = 4 * threadIdx.x; e < H; e += 4 * blockDim.x)
      atomic_add4(dst + e, smem_acc[acc_slot_of_col(e)], smem_acc[acc_slot_of_col(e + 1)], smem_acc[acc_slot_of_col(e + 2)],
                  smem_acc[acc_slot_of_col(e + 3)]);
  } else {
    for (int e = threadIdx.x; e < H; e += blockDim.x) atomicAdd(dst + e, smem_acc[acc_slot_of_col(e)]);
  }
  __syncthreads();
}

// FUSE: the gradient d_o is also the dY of the Linear that produced o (o = dropout(x W^T + b) + resid), so the same pass writes the
// 16-bit GEMM operand gT = T(d_o * keep) and adds its column sums (the bias gradient, summed over the values the weight-gradient GEMM
// reads) into dbias -- one grad_cast and one colsum launch less per LayerNorm, and d_o is not re-read twice.  keep_bits (optional): the
// dropout mask as the forward pass left it (dropout_add_layernorm), else it is regenerated from Philox.
// The three register accumulator sets cap the kernel at one 8-warp CTA per SM; at two warps per scheduler it is bound by the issue latency
// of each warp's serial instruction stream, not by its loads: prefetching a warp's next row with cp.async into a per-warp double buffer
// was measured SLOWER (72 vs 60 us per launch at 16384 x 768, profiles/train_iter12_r02.log) and is not kept; a 128-register build with
// two CTAs per SM spills the accumulators (67 us).  What does help is a shorter stream: the mask bits instead of six Philox calls per row.
template <int VPL, typename T, bool FUSE>
__global__ void __launch_bounds__(kTrThreads) layernorm_bwd_kernel(const float* __restrict__ dh, const float* __restrict__ o, int M, int H,
                                                                   const float* __restrict__ gamma, float eps, float* __restrict__ d_o,
                                                                   float* __restrict__ dgamma, float* __restrict__ dbeta, DropSpec dr,
                                                                   T* __restrict__ gT, float* __restrict__ dbias,
                                                                   const uint8_t* __restrict__ keep_bits) {
  pdl_wait();
  constexpr int NACC = FUSE ? 3 : 2;
  extern __shared__ float sacc[];  // [NACC][H]
  for (int e = threadIdx.x; e < NACC * H; e += kTrThreads) sacc[e] = 0.f;
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float ag[VPL][8], ab[VPL][8], ad[FUSE ? VPL : 1][8];
#pragma unroll
  for (int i = 0; i < VPL; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      ag[i][j] = 0.f;
      ab[i][j] = 0.f;
      if (FUSE) ad[FUSE ? i : 0][j] = 0.f;
    }
  const float keep_scale = dr.p > 0.f ? 1.0f / (1.0f - dr.p) : 1.0f;  // as drop_scales8
  for (int row = blockIdx.x * (kTrThreads / 32) + warp; row < M; row += gridDim.x * (kTrThreads / 32)) {
    float x[VPL][8], g[VPL][8];
    ld_row<float, VPL>(o + static_cast<size_t>(row) * H, lane, x);
    ld_row<float, VPL>(dh + static_cast<size_t>(row) * H, lane, g);
    uint32_t kb[VPL];
    if (FUSE && keep_bits) {
#pragma unroll
      for (int i = 0; i < VPL; ++i) kb[i] = keep_bits[static_cast<size_t>(row) * (H / 8) + i * 32 + lane];
    }
    float mean, rstd;
    stats_of<VPL>(x, H, eps, mean, rstd);
#pragma unroll
    for (int i = 0; i < VPL; ++i) {
      float w8[8];
      load8<float>(gamma + (i * 32 + lane) * 8, w8);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        x[i][j] = (x[i][j] - mean) * rstd;  // xhat
        ag[i][j] = fmaf(g[i][j], x[i][j], ag[i][j]);
        ab[i][j] += g[i][j];
        g[i][j] *= w8[j];  // dL/d(xhat)
      }
    }
    ln_bwd_core<VPL>(x, g, H, rstd);
    st_row<float, VPL>(d_o + static_cast<size_t>(row) * H, lane, g);
    if (FUSE) {
#pragma unroll
      for (int i = 0; i < VPL; ++i) {
        const size_t e0 = static_cast<size_t>(row) * H + (i * 32 + lane) * 8;
        float keep[8];
        if (keep_bits) {
#pragma unroll
          for (int j = 0; j < 8; ++j) keep[j] = (kb[i] >> j) & 1u ? keep_scale : 0.f;
        } else {
          drop_scales8(dr, e0, keep);
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          g[i][j] = to_f32<T>(from_f32<T>(g[i][j] * keep[j]));  // the value the backward GEMMs will read
          ad[FUSE ? i : 0][j] += g[i][j];
        }
        store8<T>(gT + e0, g[i]);
      }
    }
  }
  flush_feature_sums<VPL>(ag, dgamma, sacc, H, lane);
  flush_feature_sums<VPL>(ab, dbeta, sacc + H, H, lane);
  if constexpr (FUSE) flush_feature_sums<VPL>(ad, dbias, sacc + 2 * H, H, lane);
}
static int ln_bwd_grid(int M) {
  const int need = ceil_div(M, kTrThreads / 32);
  return need < 2 * num_sms() ? need : 2 * num_sms();
}
// one wave of resident CTAs (grid-stride over the rows): a second wave would only repeat the per-CTA flush of the feature sums
template <typename K>
static int ln_bwd_resident_grid(K kernel, size_t smem, int M) {
  int occ = 1;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, kTrThreads, smem) != cudaSuccess || occ < 1) occ = 1;
  const int need = ceil_div(M, kTrThreads / 32), cap = occ * num_sms();
  return need < cap ? need : cap;
}
int layernorm_bwd(const float* dh, const float* o, int M, int H, const float* gamma, float eps, float* d_o, float* dgamma, float* dbeta,
                  cudaStream_t s) {
  SD_VPL_DISPATCH(H, SD_CUDA(launch_k(layernorm_bwd_kernel<VPL, float, false>, dim3(ln_bwd_grid(M)), dim3(kTrThreads), 2 * H * sizeof(float), s, dh, o,
                                      M, H, gamma, eps, d_o, dgamma, dbeta, no_drop(), static_cast<float*>(nullptr), static_cast<float*>(nullptr),
                                      static_cast<const uint8_t*>(nullptr))));
  SD_LAUNCHED("layernorm_bwd", s);
  return SEQDIFF_OK;
}
template <typename T>
int layernorm_bwd_cast(const float* dh, const float* o, int M, int H, const float* gamma, float eps, float* d_o, float* dgamma, float* dbeta,
                       DropSpec dr, const uint8_t* keep_bits, T* gT, float* dbias, cudaStream_t s) {
  SD_CHECK(gT && dbias, "layernorm_bwd_cast: operand and bias-gradient outputs are required");
  const size_t smem = 3 * static_cast<size_t>(H) * sizeof(float);
  SD_VPL_DISPATCH(H, auto kfn = layernorm_bwd_kernel<VPL, T, true>;
                  SD_CUDA(launch_k(kfn, dim3(ln_bwd_resident_grid(kfn, smem, M)), dim3(kTrThreads), smem, s, dh, o, M, H, gamma, eps, d_o, dgamma,
                                   dbeta, dr, gT, dbias, dr.p > 0.f ? keep_bits : nullptr)));
  SD_LAUNCHED("layernorm_bwd", s);
  return SEQDIFF_OK;
}
template int layernorm_bwd_cast<bf16>(const float*, const float*, int, int, const float*, float, float*, float*, float*, DropSpec, const uint8_t*,
                                      bf16*, float*, cudaStream_t);
template int layernorm_bwd_cast<f16>(const float*, const float*, int, int, const float*, float, float*, float*, float*, DropSpec, const uint8_t*,
                                     f16*, float*, cudaStream_t);

// =====================================================================================================
// SELayer residual update backward (forward: rowwise.cu ln_modulate_kernel)
//   y = AFF ? LN(in; g, b, eps1) : in ;  n = LN0(y) (no affine, eps 1e-5) ;  out = x + gate * (n * (1 + scale) + shift)
// dout [M,H] fp32 ->  din [M,H] fp32 (gradient of `in`), optional sum_out = din + dout (gradient that reaches x through BOTH
// the residual and, for the attention update, through o = ... + x), d(shift, scale, gate) either written as T rows of dmodT
// (mod_div == 1) or atomically accumulated into dmod32 [M / mod_div, 6H] (conditioning broadcast over the graph).
// =====================================================================================================
template <typename T, int VPL, bool AFF, bool PG>
__global__ void __launch_bounds__(kTrThreads) ln_modulate_bwd_kernel(const float* __restrict__ dout, const float* __restrict__ in, int M, int H,
                                                                     const float* __restrict__ lnw, const float* __restrict__ lnb, float eps1,
                                                                     const T* __restrict__ mod, int mod_div, int chunk0, float* __restrict__ din,
                                                                     float* __restrict__ sum_out, T* __restrict__ dmodT, float* __restrict__ dmod32,
                                                                     float* __restrict__ dgamma, float* __restrict__ dbeta, int rpw) {
  pdl_wait();
  extern __shared__ float sacc[];  // [2][H] (AFF only)
  if (AFF) {
    for (int e = threadIdx.x; e < 2 * H; e += kTrThreads) sacc[e] = 0.f;
    __syncthreads();
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float ag[VPL][8], ab[VPL][8];  // (dead code without AFF)
#pragma unroll
  for (int i = 0; i < VPL; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) { ag[i][j] = 0.f; ab[i][j] = 0.f; }
  // per-graph conditioning (dmod32): a warp takes `rpw` CONSECUTIVE rows of one graph and adds their shift / scale / gate gradients in
  // registers -- one global atomic per element and warp instead of one per element and ROW (37 M contended atomics per launch at
  // 128 graphs x 128 rows before).  Per-token conditioning (dmodT): rpw = 1, the grid-stride loop over single rows as before.
  float am[PG ? 3 : 1][VPL][8];
  (void)am;
  for (int grp = blockIdx.x * (kTrThreads / 32) + warp; grp * rpw < M; grp += gridDim.x * (kTrThreads / 32)) {
  if (PG) {
#pragma unroll
    for (int c = 0; c < 3; ++c)
#pragma unroll
      for (int i = 0; i < VPL; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) am[c][i][j] = 0.f;
  }
  for (int rr = 0; rr < rpw; ++rr) {
    const int row = grp * rpw + rr;
    if (row >= M) break;
    float y[VPL][8], xh1[VPL][8], g[VPL][8];
    ld_row<float, VPL>(in + static_cast<size_t>(row) * H, lane, y);
    ld_row<float, VPL>(dout + static_cast<size_t>(row) * H, lane, g);
    float mean1 = 0.f, rstd1 = 1.f;
    if (AFF) {
      stats_of<VPL>(y, H, eps1, mean1, rstd1);
#pragma unroll
      for (int i = 0; i < VPL; ++i) {
        float w8[8], b8[8];
        load8<float>(lnw + (i * 32 + lane) * 8, w8);
        load8<float>(lnb + (i * 32 + lane) * 8, b8);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          xh1[i][j] = (y[i][j] - mean1) * rstd1;
          y[i][j] = xh1[i][j] * w8[j] + b8[j];
        }
      }
    }
    float mean0, rstd0;
    stats_of<VPL>(y, H, 1e-5f, mean0, rstd0);
    const T* mrow = mod + static_cast<size_t>(row / mod_div) * (6 * H);
#pragma unroll
    for (int i = 0; i < VPL; ++i) {
      const int e = (i * 32 + lane) * 8;
      float sh[8], sc[8], gt[8], dsh[8], dsc[8], dgt[8];
      load8<T>(mrow + (chunk0 + 0) * H + e, sh);
      load8<T>(mrow + (chunk0 + 1) * H + e, sc);
      load8<T>(mrow + (chunk0 + 2) * H + e, gt);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float n = (y[i][j] - mean0) * rstd0;
        const float go = g[i][j];
        dgt[j] = go * (n * (1.0f + sc[j]) + sh[j]);
        dsc[j] = go * gt[j] * n;
        dsh[j] = go * gt[j];
        y[i][j] = n;                              // xhat of LN0
        g[i][j] = go * gt[j] * (1.0f + sc[j]);    // dL/dn
      }
      if (dmodT) {
        T* drow = dmodT + static_cast<size_t>(row) * (6 * H);
        store8<T>(drow + (chunk0 + 0) * H + e, dsh);
        store8<T>(drow + (chunk0 + 1) * H + e, dsc);
        store8<T>(drow + (chunk0 + 2) * H + e, dgt);
      } else if constexpr (PG) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          am[0][i][j] += dsh[j];
          am[1][i][j] += dsc[j];
          am[2][i][j] += dgt[j];
        }
      }
    }
    ln_bwd_core<VPL>(y, g, H, rstd0);  // g = dL/dy
    if (AFF) {
#pragma unroll
      for (int i = 0; i < VPL; ++i) {
        float w8[8];
        load8<float>(lnw + (i * 32 + lane) * 8, w8);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          ag[i][j] = fmaf(g[i][j], xh1[i][j], ag[i][j]);
          ab[i][j] += g[i][j];
          g[i][j] *= w8[j];
        }
      }
      ln_bwd_core<VPL>(xh1, g, H, rstd1);
    }
    st_row<float, VPL>(din + static_cast<size_t>(row) * H, lane, g);
    if (sum_out) {
      float d2[VPL][8];
      ld_row<float, VPL>(dout + static_cast<size_t>(row) * H, lane, d2);
#pragma unroll
      for (int i = 0; i < VPL; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) d2[i][j] += g[i][j];
      st_row<float, VPL>(sum_out + static_cast<size_t>(row) * H, lane, d2);
    }
  }  // rows of the group
  if constexpr (PG) {
    float* drow = dmod32 + static_cast<size_t>((grp * rpw) / mod_div) * (6 * H);
#pragma unroll
    for (int c = 0; c < 3; ++c)
#pragma unroll
      for (int i = 0; i < VPL; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) atomicAdd(drow + (chunk0 + c) * H + (i * 32 + lane) * 8 + j, am[c][i][j]);
  }
  }  // groups
  if constexpr (AFF) {
    flush_feature_sums<VPL>(ag, dgamma, sacc, H, lane);
    flush_feature_sums<VPL>(ab, dbeta, sacc + H, H, lane);
  }
}
template <typename T>
int ln_modulate_bwd(const float* dout, const float* in, int M, int H, bool affine_first, const float* lnw, const float* lnb, float eps1,
                    const T* mod, int mod_div, int chunk0, float* din, float* sum_out, T* dmodT, float* dmod32, float* dgamma, float* dbeta,
                    cudaStream_t s) {
  SD_CHECK((dmodT != nullptr) != (dmod32 != nullptr), "ln_modulate_bwd: exactly one of dmodT / dmod32");
  SD_CHECK(!dmodT || mod_div == 1, "ln_modulate_bwd: direct T rows only for per-token conditioning");
  // per-graph conditioning: rows per warp = the largest of 16, 8, 4, 2, 1 that divides the rows per graph (a warp's rows share one graph)
  int rpw = 1;
  if (dmod32)
    for (int c : {16, 8, 4, 2})
      if (mod_div % c == 0) { rpw = c; break; }
  const int need = ceil_div(ceil_div(M, rpw), kTrThreads / 32);
  const int grid = need < 2 * num_sms() ? need : 2 * num_sms();
#define SD_LNMB_LAUNCH(AFF_, PG_, SMEM_)                                                                                                       \
  SD_VPL_DISPATCH(H, SD_CUDA(launch_k(ln_modulate_bwd_kernel<T, VPL, AFF_, PG_>, dim3(grid), dim3(kTrThreads), SMEM_, s, dout, in, M, H, lnw, lnb, \
                                      eps1, mod, mod_div, chunk0, din, sum_out, dmodT, dmod32, dgamma, dbeta, rpw)))
  if (affine_first) {
    if (dmod32) { SD_LNMB_LAUNCH(true, true, 2 * H * sizeof(float)); } else { SD_LNMB_LAUNCH(true, false, 2 * H * sizeof(float)); }
  } else {
    if (dmod32) { SD_LNMB_LAUNCH(false, true, 0); } else { SD_LNMB_LAUNCH(false, false, 0); }
  }
#undef SD_LNMB_LAUNCH
  SD_LAUNCHED("ln_modulate_bwd", s);
  return SEQDIFF_OK;
}
#define SD_INST_LNMB(T)                                                                                                                  \
  template int ln_modulate_bwd<T>(const float*, const float*, int, int, bool, const float*, const float*, float, const T*, int, int, float*, \
                                  float*, T*, float*, float*, float*, cudaStream_t)
SD_INST_LNMB(float);
SD_INST_LNMB(bf16);
SD_INST_LNMB(f16);

// =====================================================================================================
// BertEmbeddings backward (forward: embed_ln_multi_kernel): out = dropout(LN(x Wt + b) * g + beta) [+ te]
// dout [M,H] fp32 (gradient of `out`).  Parameter gradients only (the inputs are data): dW [H, fin] (nn.Linear layout),
// db [H], dg [H], dbeta [H].  lin = x Wt + b is recomputed (fin <= 32 multiply-adds per feature).
// =====================================================================================================
// DENSE (fin <= 8, the angle embeddings: every input feature is non-zero): dW^T[k, :] += x_k g[:] was fin * H / 32 shared atomics per
// lane and row (192 at fin = 8, H = 768 -- the launch was bound by them: ~230 us against ~20 us for the one-hot sequence embeddings).
// Instead the eight warps park their rows' g and x in shared memory, and after a barrier every THREAD owns H / 256 columns and adds
// x[w][k] * g[w][col] over the eight rows into fin * H / 256 register accumulators: plain FMAs on conflict-free reads.
template <int VPL, bool DENSE>
__global__ void __launch_bounds__(kTrThreads) embed_bwd_kernel(const float* __restrict__ dout, const float* __restrict__ x, int M, int fin, int H,
                                                               const float* __restrict__ Wt, const float* __restrict__ b,
                                                               const float* __restrict__ gamma, float eps, DropSpec dr, float* __restrict__ dW,
                                                               float* __restrict__ db, float* __restrict__ dgamma, float* __restrict__ dbeta) {
  pdl_wait();
  constexpr int NW = kTrThreads / 32;
  extern __shared__ float sacc[];  // sparse: [fin + 3][H] = dW^T rows | db | dgamma | dbeta;  DENSE: [3][H] sums | [NW][H] g rows | [NW][8] x rows
  const int n_acc = DENSE ? 3 : fin + 3, base_acc = DENSE ? 0 : fin;
  for (int e = threadIdx.x; e < n_acc * H; e += kTrThreads) sacc[e] = 0.f;
  float* sg = sacc + 3 * H;
  float* sx = sg + NW * H;
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  // db / dgamma / dbeta: every row adds to the same H columns -> per-warp register accumulators, flushed once per CTA (they were
  // 3 H of the (3 + nnz) H shared atomics per row); sparse inputs: dW^T[k, :] += x_k g[:] stays on shared atomics (k varies with the row).
  float a_db[VPL][8], a_dg[VPL][8], a_dbt[VPL][8], a_w[DENSE ? 8 : 1][VPL];
#pragma unroll
  for (int i = 0; i < VPL; ++i) {
#pragma unroll
    for (int j = 0; j < 8; ++j) { a_db[i][j] = 0.f; a_dg[i][j] = 0.f; a_dbt[i][j] = 0.f; }
#pragma unroll
    for (int k = 0; k < (DENSE ? 8 : 1); ++k) a_w[k][i] = 0.f;
  }
  // DENSE walks the rows in CTA-uniform passes of NW rows (barriers inside); the sparse form lets every warp run on its own
  for (int row0 = blockIdx.x * NW; row0 < M; row0 += gridDim.x * NW) {
    const int row = row0 + warp;
    const bool live = row < M;
    if (!DENSE && !live) break;
    float g[VPL][8];
    float xin = 0.f;
    if (live) {
      xin = lane < fin ? x[static_cast<size_t>(row) * fin + lane] : 0.f;
      float v[VPL][8];
#pragma unroll
      for (int i = 0; i < VPL; ++i) load8<float>(b + (i * 32 + lane) * 8, v[i]);
      for (int k = 0; k < fin; ++k) {
        const float xk = __shfl_sync(0xffffffffu, xin, k);
        if (xk == 0.f) continue;
#pragma unroll
        for (int i = 0; i < VPL; ++i) {
          float w8[8];
          load8<float>(Wt + static_cast<size_t>(k) * H + (i * 32 + lane) * 8, w8);
#pragma unroll
          for (int j = 0; j < 8; ++j) v[i][j] = fmaf(xk, w8[j], v[i][j]);
        }
      }
      float mean, rstd;
      stats_of<VPL>(v, H, eps, mean, rstd);
      ld_row<float, VPL>(dout + static_cast<size_t>(row) * H, lane, g);
#pragma unroll
      for (int i = 0; i < VPL; ++i) {
        float keep[8], w8[8];
        drop_scales8(dr, static_cast<size_t>(row) * H + (i * 32 + lane) * 8, keep);
        load8<float>(gamma + (i * 32 + lane) * 8, w8);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float go = g[i][j] * keep[j];
          v[i][j] = (v[i][j] - mean) * rstd;
          a_dg[i][j] = fmaf(go, v[i][j], a_dg[i][j]);
          a_dbt[i][j] += go;
          g[i][j] = go * w8[j];
        }
      }
      ln_bwd_core<VPL>(v, g, H, rstd);  // g = dL/d(lin)
#pragma unroll
      for (int i = 0; i < VPL; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) a_db[i][j] += g[i][j];
    } else {
#pragma unroll
      for (int i = 0; i < VPL; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) g[i][j] = 0.f;
    }
    if constexpr (DENSE) {
      st_row<float, VPL>(sg + static_cast<size_t>(warp) * H, lane, g);
      if (lane < 8) sx[warp * 8 + lane] = xin;  // lanes fin .. 7 hold 0
      __syncthreads();
#pragma unroll
      for (int w = 0; w < NW; ++w) {
        float xw[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) xw[k] = sx[w * 8 + k];
#pragma unroll
        for (int i = 0; i < VPL; ++i) {
          const float gv = sg[static_cast<size_t>(w) * H + i * 256 + threadIdx.x];
#pragma unroll
          for (int k = 0; k < 8; ++k) a_w[k][i] = fmaf(xw[k], gv, a_w[k][i]);
        }
      }
      __syncthreads();
    } else {
      for (int k = 0; k < fin; ++k) {
        const float xk = __shfl_sync(0xffffffffu, xin, k);
        if (xk == 0.f) continue;
#pragma unroll
        for (int i = 0; i < VPL; ++i)
#pragma unroll
          for (int j = 0; j < 8; ++j) atomicAdd(sacc + static_cast<size_t>(k) * H + acc_slot(i, lane, j), xk * g[i][j]);
      }
    }
  }
#pragma unroll
  for (int i = 0; i < VPL; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int e = acc_slot(i, lane, j);
      atomicAdd(sacc + static_cast<size_t>(base_acc) * H + e, a_db[i][j]);
      atomicAdd(sacc + (base_acc + 1) * H + e, a_dg[i][j]);
      atomicAdd(sacc + (base_acc + 2) * H + e, a_dbt[i][j]);
    }
  __syncthreads();
  // dW is [H, fin] (nn.Linear layout): the fin values of one output column are contiguous
  const bool w4 = aligned16(dW) && fin % 4 == 0;
  if constexpr (DENSE) {
#pragma unroll
    for (int i = 0; i < VPL; ++i) {
      float* col = dW + static_cast<size_t>(i * 256 + threadIdx.x) * fin;
      if (w4 && fin == 8) {
        atomic_add4(col, a_w[0][i], a_w[1][i], a_w[2][i], a_w[3][i]);
        atomic_add4(col + 4, a_w[4][i], a_w[5][i], a_w[6][i], a_w[7][i]);
      } else {
#pragma unroll
        for (int k = 0; k < 8; ++k)
          if (k < fin && a_w[k][i] != 0.f) atomicAdd(col + k, a_w[k][i]);
      }
    }
  } else if (w4) {
    const int q = fin / 4;  // groups of four input features per output column
    for (int e = threadIdx.x; e < q * H; e += kTrThreads) {
      const int h = e / q, k = (e - h * q) * 4, sl = acc_slot_of_col(h);
      const float v0 = sacc[k * H + sl], v1 = sacc[(k + 1) * H + sl], v2 = sacc[(k + 2) * H + sl], v3 = sacc[(k + 3) * H + sl];
      if (v0 != 0.f || v1 != 0.f || v2 != 0.f || v3 != 0.f) atomic_add4(dW + static_cast<size_t>(h) * fin + k, v0, v1, v2, v3);
    }
  } else {
    for (int e = threadIdx.x; e < fin * H; e += kTrThreads) {
      const int k = e / H, h = e - k * H;
      const float v = sacc[k * H + acc_slot_of_col(h)];
      if (v != 0.f) atomicAdd(dW + static_cast<size_t>(h) * fin + k, v);
    }
  }
  if (aligned16(db) && aligned16(dgamma) && aligned16(dbeta)) {
    for (int e = 4 * threadIdx.x; e < H; e += 4 * kTrThreads) {
      const int s0 = acc_slot_of_col(e), s1 = acc_slot_of_col(e + 1), s2 = acc_slot_of_col(e + 2), s3 = acc_slot_of_col(e + 3);
      atomic_add4(db + e, sacc[base_acc * H + s0], sacc[base_acc * H + s1], sacc[base_acc * H + s2], sacc[base_acc * H + s3]);
      atomic_add4(dgamma + e, sacc[(base_acc + 1) * H + s0], sacc[(base_acc + 1) * H + s1], sacc[(base_acc + 1) * H + s2], sacc[(base_acc + 1) * H + s3]);
      atomic_add4(dbeta + e, sacc[(base_acc + 2) * H + s0], sacc[(base_acc + 2) * H + s1], sacc[(base_acc + 2) * H + s2], sacc[(base_acc + 2) * H + s3]);
    }
  } else {
    for (int e = threadIdx.x; e < H; e += kTrThreads) {
      const int sl = acc_slot_of_col(e);
      atomicAdd(db + e, sacc[base_acc * H + sl]);
      atomicAdd(dgamma + e, sacc[(base_acc + 1) * H + sl]);
      atomicAdd(dbeta + e, sacc[(base_acc + 2) * H + sl]);
    }
  }
}
int embed_bwd(const float* dout, const float* x, int M, int fin, int H, const float* Wt, const float* b, const float* gamma, float eps, DropSpec dr,
              float* dW, float* db, float* dgamma, float* dbeta, cudaStream_t s) {
  SD_CHECK(fin >= 1 && fin <= 32, "embed_bwd: fin in [1,32]");
  const int need = ceil_div(M, kTrThreads / 32);
  const int grid = need < num_sms() ? need : num_sms();
  const bool dense = fin <= 8;  // the one-hot sequence embeddings (fin = 20) take the shared-atomic form
  const size_t smem = dense ? (static_cast<size_t>(3 + kTrThreads / 32) * H + (kTrThreads / 32) * 8) * sizeof(float)
                            : static_cast<size_t>(fin + 3) * H * sizeof(float);
#define SD_EB_LAUNCH_(DENSE_)                                                                                       \
  {                                                                                                                 \
    auto kfn = embed_bwd_kernel<VPL, DENSE_>;                                                                       \
    static bool configured = false;                                                                                 \
    if (!configured) {                                                                                              \
      SD_CUDA(cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, 35 * 1024 * 4));               \
      configured = true;                                                                                            \
    }                                                                                                               \
    SD_CUDA(launch_k(kfn, dim3(grid), dim3(kTrThreads), smem, s, dout, x, M, fin, H, Wt, b, gamma, eps, dr, dW, db, dgamma, dbeta)); \
  }
#define SD_EB_LAUNCH() if (dense) SD_EB_LAUNCH_(true) else SD_EB_LAUNCH_(false)
  SD_VPL_DISPATCH(H, SD_EB_LAUNCH());
#undef SD_EB_LAUNCH_
#undef SD_EB_LAUNCH
  SD_LAUNCHED("embed_bwd", s);
  return SEQDIFF_OK;
}

// =====================================================================================================
// AminoAcidPredictor tail backward (forward: predictor_tail_kernel): logits = LN(y; g, b) W2^T + b2
// dlogits [M,F] fp32 -> dy [M,H] fp32; dW2 [F,H], db2 [F], dg [H], db [H] accumulated.
// =====================================================================================================
// F == 20 (the amino-acid head; seqdiff_train_step requires it).  A warp per row accumulating dW2 through F * H / 32 = 480 shared atomics
// per lane was bound by them (284 us per launch at 16384 rows).  Here the eight warps of a CTA park LN(y) and dlogits of their rows in
// shared memory, and after a barrier every THREAD owns H / 256 columns of dW2 for all 20 classes in registers (60 accumulators, plain FMAs
// on conflict-free reads); dgamma / dbeta accumulate in per-warp registers and meet once per CTA (flush_feature_sums).
template <typename T, int VPL>
__global__ void __launch_bounds__(kTrThreads) predictor_tail_bwd20_kernel(const float* __restrict__ dlogits, const T* __restrict__ y, int M, int H,
                                                                          const float* __restrict__ gamma, const float* __restrict__ beta, float eps,
                                                                          const float* __restrict__ W2, float* __restrict__ dy,
                                                                          float* __restrict__ dW2, float* __restrict__ db2, float* __restrict__ dgamma,
                                                                          float* __restrict__ dbeta) {
  pdl_wait();
  constexpr int F = 20, NW = kTrThreads / 32;
  extern __shared__ float smem[];
  float* sW = smem;                                   // [F][H]   W2
  float* sG = sW + static_cast<size_t>(F) * H;        // [2][H]   dgamma | dbeta (flush)
  float* sln = sG + 2 * H;                            // [NW][H]  LN(y) rows of the current pass
  float* sdl = sln + static_cast<size_t>(NW) * H;     // [NW][32] dlogits rows of the current pass (zero = dead row / lane >= F)
  float* sB = sdl + NW * 32;                          // [32]     db2
  for (int i = threadIdx.x; i < F * H; i += kTrThreads) sW[i] = W2[i];
  for (int i = threadIdx.x; i < 2 * H; i += kTrThreads) sG[i] = 0.f;
  if (threadIdx.x < 32) sB[threadIdx.x] = 0.f;
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float a_w[F][VPL], ag[VPL][8], ab[VPL][8];
#pragma unroll
  for (int i = 0; i < VPL; ++i) {
#pragma unroll
    for (int f = 0; f < F; ++f) a_w[f][i] = 0.f;
#pragma unroll
    for (int j = 0; j < 8; ++j) { ag[i][j] = 0.f; ab[i][j] = 0.f; }
  }
  for (int row0 = blockIdx.x * NW; row0 < M; row0 += gridDim.x * NW) {  // CTA-uniform passes of NW rows (barriers inside)
    const int row = row0 + warp;
    float dl = 0.f;
    if (row < M) {
      float v[VPL][8], g[VPL][8], ln[VPL][8];
      ld_row<T, VPL>(y + static_cast<size_t>(row) * H, lane, v);
      float mean, rstd;
      stats_of<VPL>(v, H, eps, mean, rstd);
      dl = lane < F ? dlogits[static_cast<size_t>(row) * F + lane] : 0.f;
      if (dl != 0.f) atomicAdd(sB + lane, dl);
#pragma unroll
      for (int i = 0; i < VPL; ++i) {
        float w8[8], b8[8];
        load8<float>(gamma + (i * 32 + lane) * 8, w8);
        load8<float>(beta + (i * 32 + lane) * 8, b8);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          v[i][j] = (v[i][j] - mean) * rstd;
          ln[i][j] = v[i][j] * w8[j] + b8[j];
          g[i][j] = 0.f;
        }
      }
      const bool any = __ballot_sync(0xffffffffu, dl != 0.f) != 0u;  // rows outside the noised set carry a zero gradient: skipped entirely
      if (any) {
        st_row<float, VPL>(sln + static_cast<size_t>(warp) * H, lane, ln);
        for (int f = 0; f < F; ++f) {
          const float d = __shfl_sync(0xffffffffu, dl, f);
          if (d == 0.f) continue;
#pragma unroll
          for (int i = 0; i < VPL; ++i) {
            float w8[8];
            load8<float>(sW + static_cast<size_t>(f) * H + (i * 32 + lane) * 8, w8);
#pragma unroll
            for (int j = 0; j < 8; ++j) g[i][j] = fmaf(d, w8[j], g[i][j]);
          }
        }
#pragma unroll
        for (int i = 0; i < VPL; ++i) {
          float w8[8];
          load8<float>(gamma + (i * 32 + lane) * 8, w8);
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            ag[i][j] = fmaf(g[i][j], v[i][j], ag[i][j]);
            ab[i][j] += g[i][j];
            g[i][j] *= w8[j];
          }
        }
        ln_bwd_core<VPL>(v, g, H, rstd);
      }
      st_row<float, VPL>(dy + static_cast<size_t>(row) * H, lane, g);
    }
    sdl[warp * 32 + lane] = dl;
    __syncthreads();
#pragma unroll 1
    for (int w = 0; w < NW; ++w) {
      float lnv[VPL];
      bool live = false;
      float d[F];
#pragma unroll
      for (int f = 0; f < F; ++f) {
        d[f] = sdl[w * 32 + f];
        live = live || d[f] != 0.f;
      }
      if (!live) continue;  // CTA-uniform (shared values): its sln row may be stale
#pragma unroll
      for (int i = 0; i < VPL; ++i) lnv[i] = sln[static_cast<size_t>(w) * H + i * 256 + threadIdx.x];
#pragma unroll
      for (int f = 0; f < F; ++f)
#pragma unroll
        for (int i = 0; i < VPL; ++i) a_w[f][i] = fmaf(d[f], lnv[i], a_w[f][i]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int f = 0; f < F; ++f)
#pragma unroll
    for (int i = 0; i < VPL; ++i)
      if (a_w[f][i] != 0.f) atomicAdd(dW2 + static_cast<size_t>(f) * H + i * 256 + threadIdx.x, a_w[f][i]);
  flush_feature_sums<VPL>(ag, dgamma, sG, H, lane);
  flush_feature_sums<VPL>(ab, dbeta, sG + H, H, lane);
  if (threadIdx.x < F) atomicAdd(db2 + threadIdx.x, sB[threadIdx.x]);
}
template <typename T>
int predictor_tail_bwd(const float* dlogits, const T* y, int M, int H, const float* gamma, const float* beta, float eps, const float* W2, int F,
                       float* dy, float* dW2, float* db2, float* dgamma, float* dbeta, cudaStream_t s) {
  SD_CHECK(F == 20, "predictor_tail_bwd: feature_size must be 20");
  const int need = ceil_div(M, kTrThreads / 32);
  const int grid = need < num_sms() ? need : num_sms();
  const size_t smem = (static_cast<size_t>(20 + 2 + kTrThreads / 32) * H + (kTrThreads / 32) * 32 + 32) * sizeof(float);
#define SD_PTB20_LAUNCH()                                                                                            \
  {                                                                                                                  \
    auto kfn = predictor_tail_bwd20_kernel<T, VPL>;                                                                  \
    static bool configured = false;                                                                                  \
    if (!configured) {                                                                                               \
      SD_CUDA(cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));                   \
      configured = true;                                                                                             \
    }                                                                                                                \
    SD_CUDA(launch_k(kfn, dim3(grid), dim3(kTrThreads), smem, s, dlogits, y, M, H, gamma, beta, eps, W2, dy, dW2, db2, dgamma, dbeta)); \
  }
  SD_VPL_DISPATCH(H, SD_PTB20_LAUNCH());
#undef SD_PTB20_LAUNCH
  SD_LAUNCHED("predictor_tail_bwd", s);
  return SEQDIFF_OK;
}
template int predictor_tail_bwd<float>(const float*, const float*, int, int, const float*, const float*, float, const float*, int, float*, float*,
                                       float*, float*, float*, cudaStream_t);
template int predictor_tail_bwd<bf16>(const float*, const bf16*, int, int, const float*, const float*, float, const float*, int, float*, float*,
                                      float*, float*, float*, cudaStream_t);
template int predictor_tail_bwd<f16>(const float*, const f16*, int, int, const float*, const float*, float, const float*, int, float*, float*,
                                     float*, float*, float*, cudaStream_t);

// =====================================================================================================
// loss gradient: total = CE_mean(noised rows) + elbo_loss(noised rows)   (model.py:330-344, utils.py:132-161)
// With p = softmax(z), H = -sum p log p, y = one-hot target, q = softmax(one-hot target), N = #noised rows:
//   dz = [ (p - y) + (p - q) - p * (log p + H) ] / N      on noised rows, 0 elsewhere.
// (log_softmax(z + 1e-6) = log_softmax(z) analytically; the eps shift has no gradient.)  N is read from the loss-terms buffer
// written by loss_terms() on the same stream (terms[1]).
// =====================================================================================================
__global__ void __launch_bounds__(256) loss_bwd_kernel(int N, const float* __restrict__ logits, const float* __restrict__ x0,
                                                       const float* __restrict__ x_t, const double* __restrict__ terms, float* __restrict__ dlogits) {
  pdl_wait();
  constexpr int C = SEQDIFF_NUM_CLASSES;
  const double n_noised = terms[1];
  const float inv_n = n_noised > 0.0 ? static_cast<float>(1.0 / n_noised) : 0.f;
  for (int n = blockIdx.x * 256 + threadIdx.x; n < N; n += gridDim.x * 256) {
    float z[C], a[C], b[C];
#pragma unroll
    for (int j4 = 0; j4 < C; j4 += 4) {
      const float4 v = *reinterpret_cast<const float4*>(logits + static_cast<size_t>(n) * C + j4);
      const float4 u = *reinterpret_cast<const float4*>(x0 + static_cast<size_t>(n) * C + j4);
      const float4 w = *reinterpret_cast<const float4*>(x_t + static_cast<size_t>(n) * C + j4);
      z[j4] = v.x; z[j4 + 1] = v.y; z[j4 + 2] = v.z; z[j4 + 3] = v.w;
      a[j4] = u.x; a[j4 + 1] = u.y; a[j4 + 2] = u.z; a[j4 + 3] = u.w;
      b[j4] = w.x; b[j4 + 1] = w.y; b[j4 + 2] = w.z; b[j4 + 3] = w.w;
    }
    int tgt = 0, xt = 0;
#pragma unroll
    for (int j = 1; j < C; ++j) {
      if (a[j] > a[tgt]) tgt = j;
      if (b[j] > b[xt]) xt = j;
    }
    float out[C];
    if (xt != tgt) {
      float mx = z[0];
#pragma unroll
      for (int j = 1; j < C; ++j) mx = fmaxf(mx, z[j]);
      float sum = 0.f;
#pragma unroll
      for (int j = 0; j < C; ++j) sum += expf(z[j] - mx);
      const float lse = logf(sum);
      float amax = a[0];
#pragma unroll
      for (int j = 1; j < C; ++j) amax = fmaxf(amax, a[j]);
      float qs = 0.f, q[C];
#pragma unroll
      for (int j = 0; j < C; ++j) { q[j] = expf(a[j] - amax); qs += q[j]; }
      float ent = 0.f, p[C], lp[C];
#pragma unroll
      for (int j = 0; j < C; ++j) {
        lp[j] = z[j] - mx - lse;
        p[j] = expf(lp[j]);
        ent -= p[j] * lp[j];
      }
#pragma unroll
      for (int j = 0; j < C; ++j) out[j] = ((p[j] - (j == tgt ? 1.f : 0.f)) + (p[j] - q[j] / qs) - p[j] * (lp[j] + ent)) * inv_n;
    } else {
#pragma unroll
      for (int j = 0; j < C; ++j) out[j] = 0.f;
    }
#pragma unroll
    for (int j4 = 0; j4 < C; j4 += 4)
      *reinterpret_cast<float4*>(dlogits + static_cast<size_t>(n) * C + j4) = make_float4(out[j4], out[j4 + 1], out[j4 + 2], out[j4 + 3]);
  }
}
int loss_bwd(int N, const float* logits, const float* x0, const float* x_t, const double* terms, float* dlogits, cudaStream_t s) {
  SD_CHECK(N > 0, "empty loss");
  SD_CUDA(launch_k(loss_bwd_kernel, dim3(ceil_div(N, 256)), dim3(256), 0, s, N, logits, x0, x_t, terms, dlogits));
  SD_LAUNCHED("loss_bwd", s);
  return SEQDIFF_OK;
}

// =====================================================================================================
// optimizer: global-norm clip + AdamW on the flat (gradient, m, v) buffers and the fp32 master parameters
// =====================================================================================================
// sum of squares of the flat gradient, fp64 accumulation, fixed-order fold by the last CTA
__global__ void __launch_bounds__(256) sumsq_kernel(const float* __restrict__ g, size_t n, double* __restrict__ partial, unsigned* __restrict__ arrive,
                                                    double* __restrict__ out) {
  pdl_wait();
  double acc = 0.0;
  const size_t n4 = n / 4;
  // four independent 16-byte loads per thread and pass: 2 CTAs x 256 threads per SM with one load each keep ~1 MB in flight on the whole
  // part, a fifth of what the HBM latency needs
  const size_t stride = static_cast<size_t>(gridDim.x) * 256;
  size_t i = static_cast<size_t>(blockIdx.x) * 256 + threadIdx.x;
  for (; i + 3 * stride < n4; i += 4 * stride) {
    float4 v[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) v[u] = *reinterpret_cast<const float4*>(g + 4 * (i + u * stride));
#pragma unroll
    for (int u = 0; u < 4; ++u)
      acc += static_cast<double>(v[u].x) * v[u].x + static_cast<double>(v[u].y) * v[u].y + static_cast<double>(v[u].z) * v[u].z +
             static_cast<double>(v[u].w) * v[u].w;
  }
  for (; i < n4; i += stride) {
    const float4 v = *reinterpret_cast<const float4*>(g + 4 * i);
    acc += static_cast<double>(v.x) * v.x + static_cast<double>(v.y) * v.y + static_cast<double>(v.z) * v.z + static_cast<double>(v.w) * v.w;
  }
  if (blockIdx.x == 0 && threadIdx.x < n - 4 * n4) {
    const float v = g[4 * n4 + threadIdx.x];
    acc += static_cast<double>(v) * v;
  }
  __shared__ double sw[8];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0) sw[threadIdx.x >> 5] = acc;
  __syncthreads();
  __shared__ bool last;
  if (threadIdx.x == 0) {
    double v = 0.0;
    for (int w = 0; w < 8; ++w) v += sw[w];
    partial[blockIdx.x] = v;
    __threadfence();
    last = atomicAdd(arrive, 1u) == gridDim.x - 1;
  }
  __syncthreads();
  if (last && threadIdx.x == 0) {
    __threadfence();
    double v = 0.0;
    for (unsigned c = 0; c < gridDim.x; ++c) v += reinterpret_cast<const volatile double*>(partial)[c];
    *out = v;
    *arrive = 0u;
  }
}

struct AdamSlots {  // device table: one entry per parameter tensor
  float* const* w;        // [n] master weights
  const int64_t* off;     // [n + 1] offsets into the flat buffers
  int n;
};
// one CTA-stride pass over the flat index space in groups of four consecutive elements; the tensor of a group is found by binary search
// in `off`.  A group that lies inside one tensor and whose master pointer is 16 B aligned moves as float4 (g, m, v, w: 4 loads + 3 stores
// of 16 B); a group that straddles a tensor boundary (or an unaligned tensor) takes the scalar path element by element.  Same arithmetic
// per element on both paths.
__device__ __forceinline__ void adamw_one(float& p, float& mi, float& vi, float gi, float lr, float beta1, float beta2, float eps, float wd,
                                          float bc1, float rs_bc2) {
  p *= 1.0f - lr * wd;                       // decoupled weight decay (torch.optim.AdamW)
  mi = beta1 * mi + (1.0f - beta1) * gi;
  vi = beta2 * vi + (1.0f - beta2) * gi * gi;
  const float denom = sqrtf(vi) / rs_bc2 + eps;
  p -= (lr / bc1) * (mi / denom);
}
__global__ void __launch_bounds__(256) adamw_kernel(AdamSlots sl, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v,
                                                    size_t total, const double* __restrict__ sumsq, float grad_scale, float max_norm, float lr,
                                                    float beta1, float beta2, float eps, float wd, float bc1, float bc2, float* __restrict__ norm_out) {
  pdl_wait();
  // torch.nn.utils.clip_grad_norm_: coef = max_norm / (total_norm + 1e-6), clamped to 1
  const float total_norm = sqrtf(static_cast<float>(*sumsq)) * grad_scale;
  float coef = 1.0f;
  if (max_norm > 0.f) coef = fminf(max_norm / (total_norm + 1e-6f), 1.0f);
  if (norm_out && blockIdx.x == 0 && threadIdx.x == 0) *norm_out = total_norm;
  const float gs = grad_scale * coef;
  const float rs_bc2 = sqrtf(bc2);
  const size_t groups = (total + 3) / 4;
  for (size_t q = static_cast<size_t>(blockIdx.x) * 256 + threadIdx.x; q < groups; q += static_cast<size_t>(gridDim.x) * 256) {
    const size_t i = 4 * q;
    int lo = 0, hi = sl.n;  // off[lo] <= i < off[hi]
    while (hi - lo > 1) {
      const int mid = (lo + hi) >> 1;
      if (static_cast<size_t>(__ldg(sl.off + mid)) <= i) lo = mid; else hi = mid;
    }
    float* w = sl.w[lo] + (i - static_cast<size_t>(sl.off[lo]));
    if (i + 4 <= static_cast<size_t>(sl.off[lo + 1]) && (reinterpret_cast<uintptr_t>(w) & 15) == 0) {
      const float4 g4 = *reinterpret_cast<const float4*>(g + i);
      float4 m4 = *reinterpret_cast<const float4*>(m + i), v4 = *reinterpret_cast<const float4*>(v + i), p4 = *reinterpret_cast<const float4*>(w);
      adamw_one(p4.x, m4.x, v4.x, g4.x * gs, lr, beta1, beta2, eps, wd, bc1, rs_bc2);
      adamw_one(p4.y, m4.y, v4.y, g4.y * gs, lr, beta1, beta2, eps, wd, bc1, rs_bc2);
      adamw_one(p4.z, m4.z, v4.z, g4.z * gs, lr, beta1, beta2, eps, wd, bc1, rs_bc2);
      adamw_one(p4.w, m4.w, v4.w, g4.w * gs, lr, beta1, beta2, eps, wd, bc1, rs_bc2);
      *reinterpret_cast<float4*>(m + i) = m4;
      *reinterpret_cast<float4*>(v + i) = v4;
      *reinterpret_cast<float4*>(w) = p4;
    } else {
      for (size_t e = i; e < i + 4 && e < total; ++e) {
        while (e >= static_cast<size_t>(sl.off[lo + 1])) ++lo;  // zero-sized tensors are skipped too
        float* we = sl.w[lo] + (e - static_cast<size_t>(sl.off[lo]));
        float p = *we, mi = m[e], vi = v[e];
        adamw_one(p, mi, vi, g[e] * gs, lr, beta1, beta2, eps, wd, bc1, rs_bc2);
        m[e] = mi;
        v[e] = vi;
        *we = p;
      }
    }
  }
}
int adamw_step(float* const* d_w, const int64_t* d_off, int n_slots, size_t total, const float* g, float* m, float* v, float grad_scale,
               float max_norm, float lr, float beta1, float beta2, float eps, float wd, int step, double* d_scratch, float* norm_out, cudaStream_t s) {
  SD_CHECK(step >= 1 && total > 0, "adamw: step counts from 1");
  SD_CHECK(((reinterpret_cast<uintptr_t>(g) | reinterpret_cast<uintptr_t>(m) | reinterpret_cast<uintptr_t>(v)) & 15) == 0,
           "flat gradient / moment buffers must be 16 B aligned");
  const int ctas = 2 * num_sms();
  unsigned* arrive = reinterpret_cast<unsigned*>(d_scratch + ctas + 1);
  SD_CUDA(launch_k(sumsq_kernel, dim3(ctas), dim3(256), 0, s, g, total, d_scratch + 1, arrive, d_scratch));
  SD_LAUNCHED("grad_sumsq", s);
  const float bc1 = 1.0f - powf(beta1, static_cast<float>(step)), bc2 = 1.0f - powf(beta2, static_cast<float>(step));
  AdamSlots sl{d_w, d_off, n_slots};
  SD_CUDA(launch_k(adamw_kernel, dim3(8 * num_sms()), dim3(256), 0, s, sl, g, m, v, total, d_scratch, grad_scale, max_norm, lr, beta1, beta2, eps, wd,
                   bc1, bc2, norm_out));
  SD_LAUNCHED("adamw", s);
  return SEQDIFF_OK;
}

}  // namespace seqdiff
